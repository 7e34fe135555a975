// ssb_solver.cuh - generic solver bodies: one CUDA thread = one problem.
//
//   layer_problem_sw / _lw : one (column, interval, layer): Gamma matrices and
//       layer transfer matrices -> layer scratch
//       (radsurf_urban_sw.F90:335-585, radsurf_urban_lw.F90:296-546 and the
//        forest equivalents)
//   column_sweeps_sw / _lw : one (column, interval): upward adding sweep,
//       boundary conditions out, the two downward passes and the flux
//       partition (radsurf_urban_sw.F90:591-984, radsurf_urban_lw.F90:552-858)
//   surface_column        : Flat tiles (radsurf_interface.F90:122-173) and the
//       single-layer urban models (radsurf_simple_urban_sw/lw.F90)
//
// The bodies are SSB_HD so that tests can run the identical code on the host;
// the kernels in ssb_kernels.cu are thin index wrappers around them.
//
// Scratch layout (device, per chunk of columns): problems q = column_in_chunk *
// nspec + interval are tiled by kScratchTile = 128 (one thread block of the sweep
// kernels); element e of level l of problem q lives at
//   base[(((q / 128) * nlev + l) * nelem + e) * 128 + q % 128],
// i.e. adjacent threads touch adjacent doubles in every access and, for a given
// problem and level, element e sits at the compile-time offset e * 128 doubles, so
// the register-resident kernels address a whole layer from one base pointer.
#pragma once
#include "../../include/spartacus_b200.h"
#include "ssb_geometry.cuh"
#include "ssb_radtool.cuh"

namespace ssb {

struct LgTable {  // legendre_gauss_type, radtool_legendre_gauss.F90:25-48
  int ns;
  double mu[SSB200_MAX_NSTREAM], tan_ang[SSB200_MAX_NSTREAM], weight[SSB200_MAX_NSTREAM];
  double hweight[SSB200_MAX_NSTREAM], vweight[SSB200_MAX_NSTREAM];
  double vadjustment, vadjustment2;
};

struct ClassArgs {
  SolveCfg cfg;
  LgTable lg;
  // columns of this launch
  int ncols;        // columns in this chunk
  int lmax;         // max layers of a column in this chunk
  const int *cols;  // [ncols] 0-based global column index
  const int *nlay, *istartlay;  // global per-column arrays (istartlay 1-based)
  ssb200_canopy_properties cp;       // device pointers (double members)
  ssb200_sw_spectral_properties sw;  // device pointers
  ssb200_lw_spectral_properties lw;  // device pointers
  int use_sw_direct_albedo;
  ssb200_boundary_conds_out bc;
  ssb200_canopy_flux f1, f2;  // SW: norm_dir, norm_diff ; LW: internal, norm
  double *layer;              // layer-matrix scratch (ne_layer elements x lmax levels)
  double *sweep;              // interface scratch (ne_sweep elements x lmax+1 levels)
  int ne_layer, ne_sweep;
  int ne_layer_geo;           // first element of the geometry block in the layer scratch
  int *perm;                  // fast path: layer problems grouped by solved sub-block (3 segments of nt)
  int *perm_count;            // [3] problems per segment
  int *status;                // failure counter
  // column-resident ("fused") path: `layer` is a set of PRIVATE one-level tiles, one per thread
  // block (re-used for every layer of every column the block solves, so it stays in L2), and
  // `sweep` holds the per-level down-pass operator records (ssb_fused.cuh)
  int fused;
  int save_profile;           // flux profiles requested (decides whether their operator rows are formed)
  // Level-major staging of the per-layer arrays (register-resident path; ssb_driver.hpp): 0 = the
  // per-layer members of cp / sw / lw / f1 / f2 are the caller's arrays in the reference layout
  // (packed ragged layers, istartlay); > 0 = they are the chunk's staging buffers, where layer `lev`
  // of chunk column ic sits at index ic + lev * lstride (lstride = columns of the chunk), so that the
  // threads of a warp (neighbouring columns, one level) touch consecutive addresses.
  int lstride;
};

// index of layer `lev` of chunk column ic (global column col) in the per-layer arrays, and the index
// distance between vertically adjacent layers of a column (see ClassArgs::lstride)
SSB_HDI int layer_index(const ClassArgs &a, int ic, int col, int lev) {
  return a.lstride ? ic + lev * a.lstride : a.istartlay[col] - 1 + lev;
}
SSB_HDI int layer_step(const ClassArgs &a) { return a.lstride ? a.lstride : 1; }

constexpr int kScratchTile = 128;
SSB_HDI size_t sidx(int e, int lev, int nlev, int nelem, int q) {
  return (((size_t)(q / kScratchTile) * (size_t)nlev + (size_t)lev) * (size_t)nelem + (size_t)e) * kScratchTile +
         (size_t)(q % kScratchTile);
}
// Layer scratch of problem q: per (tile, level) in the split path; in the fused path the tile of the
// calling thread block (slot = blockIdx.x on the device, 0 in the serial host build), one level.
SSB_HDI size_t layer_sidx(const ClassArgs &a, int e, int lev, int q) {
  if (a.fused) {
#if defined(__CUDA_ARCH__)
    const size_t slot = blockIdx.x;
#else
    const size_t slot = 0;
#endif
    return (slot * (size_t)a.ne_layer + (size_t)e) * kScratchTile + (size_t)(q % kScratchTile);
  }
  return sidx(e, lev, a.lmax, a.ne_layer, q);
}
// doubles of a scratch area of `nelem` elements x `nlev` levels for `width` problems
SSB_HDI size_t scratch_doubles(size_t nelem, size_t nlev, size_t width) {
  return ((width + kScratchTile - 1) / kScratchTile) * kScratchTile * nelem * nlev;
}

// element counts of the two scratch areas.  The layer area ends with a geometry block
// written before the layer kernels run (register-resident path): f_wall[3], od_scaling[3],
// f_wall_dir_clear, the solved sub-block ("segment": 0 all regions, 1 clear region only,
// 2 vegetated regions only), frac[3], the six exchange rates and norm_perim_wall[3]: the
// layer geometry is evaluated once per layer, the layer kernels and the sweeps read it, and
// the sweeps skip the structural zeros of partially solved layers.
constexpr int kGeoElems = 20;
// entries [to + 3*from] of f_exchange that can be non-zero: 1, 2, 3, 5, 6, 7
SSB_HDI int geo_exchange_index(int i) { return i < 3 ? i + 1 : i + 2; }
SSB_HDI int sw_layer_elems(int n, int d) { return 3 * n * n + 3 * n * d + 2 * d * d + kGeoElems; }
SSB_HDI int lw_layer_elems(int n, int nreg) { return 3 * n * n + 2 * n + 3 * nreg + 1 + kGeoElems; }
SSB_HDI int sw_sweep_elems(int n, int d, int m, int db, int nreg, int nrb) {
  return 2 * n * n + n * d + m * m + m * db + 2 * nreg * nrb;
}
SSB_HDI int lw_sweep_elems(int n, int m, int nreg, int nrb) { return 2 * n * n + n + m * m + m + 2 * nreg * nrb; }
// interface scratch of the register-resident sweeps: a_above and d_above / source_above per level
// (SwSweepLayout / LwSweepLayout::state_doubles, ssb_fast_sweeps.cuh)
SSB_HD constexpr int fast_sw_sweep_elems(int n, int d) { return n * n + n * d; }
SSB_HD constexpr int fast_lw_sweep_elems(int n) { return n * n + n; }

#define SSB_LAY(arr, g, il) (arr[(size_t)(g) + (size_t)nspec * (size_t)(il)])

SSB_HDI void count_failure(int *status, int nfail) {
  if (nfail == 0 || status == nullptr) return;
#if defined(__CUDA_ARCH__)
  atomicAdd(status, nfail);
#else
  *status += nfail;
#endif
}

// ---------------------------------------------------------------------------
// Layer problems
// ---------------------------------------------------------------------------
template <int NS>
SSB_HD inline void layer_problem_sw(const ClassArgs &a, int q, int lev) {
  constexpr int NC = 3 * NS;
  const SolveCfg &c = a.cfg;
  const int nspec = c.nspec, nreg = c.nreg, ns = c.ns, n = nreg * ns;
  const int ic = q / nspec, g = q % nspec;
  const int col = a.cols[ic];
  if (lev >= a.nlay[col]) return;
  const double cos_sza = a.cp.cos_sza[col];
  if (!(cos_sza > 0.0)) return;
  const int il = a.istartlay[col] - 1 + lev;
  const int width = a.ne_layer;  // element count of the layer scratch (sidx)
  const double zcos = c.urban ? dmax(cos_sza, 1.0e-6) : cos_sza;
  double sin0 = 0.0, tan0;
  if (c.urban) {
    sin0 = sqrt(1.0 - zcos * zcos);
    tan0 = sin0 / zcos;
  } else {
    tan0 = sqrt(1.0 - cos_sza * cos_sza) / dmax(cos_sza, 1.0e-6);
  }
  const double bf = c.urban ? a.cp.building_fraction[il] : 0.0;
  const double bs = c.urban ? a.cp.building_scale[il] : 0.0;
  const bool veg = nreg > 1 || !c.urban;
  const double vf = (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il] : 0.0;
  const double vs = (veg && a.cp.veg_scale) ? a.cp.veg_scale[il] : 1.0;
  const double ve = (veg && a.cp.veg_ext) ? a.cp.veg_ext[il] : 0.0;
  const double vcf = (c.urban && nreg > 1 && a.cp.veg_contact_fraction) ? a.cp.veg_contact_fraction[il] : 0.0;
  const double vfsd = (nreg == 3) ? a.cp.veg_fsd[il] : 0.0;
  LayerGeom gm;
  layer_geometry(c, bf, bs, vf, vs, vcf, vfsd, 1.0, gm);

  double ext[3], ssa[3];
  ext[0] = SSB_LAY(a.sw.air_ext, g, il);
  ssa[0] = SSB_LAY(a.sw.air_ssa, g, il);
  for (int r = 1; r < nreg; ++r) {
    const double vssa = SSB_LAY(a.sw.veg_ssa, g, il);
    const double od = (nreg == 2) ? 1.0 : gm.od_scaling[r];
    if (nreg == 2) {
      ext[r] = ext[0] + ve;
      ssa[r] = (ext[0] * ssa[0] + ve * vssa) / dmax(ext[r], 1.0e-8);
    } else {
      ext[r] = ext[0] + od * ve;
      ssa[r] = (ext[0] * ssa[0] + od * ve * vssa) / dmax(ext[r], 1.0e-8);
    }
  }
  double wall_ext = 0.0, wall_factor = 0.0;
  if (c.urban) {
    const double wa = SSB_LAY(a.sw.wall_albedo, g, il), wsf = SSB_LAY(a.sw.wall_specular_frac, g, il);
    wall_ext = 1.0 - wa * wsf;
    wall_factor = wa * (1.0 - wsf);
  }
  // Gamma matrices of the solved sub-block only (regions r0 .. r0+nr-1); the
  // entries coupling to unsolved regions are not used by the reference either
  // (it passes array sections, urban_sw:526-553).
  const int r0 = gm.r0, nr = gm.nr, nn = nr * ns;
  double g0[9], g1[NC * NC], g2[NC * NC], g3[NC * 3];
  for (int i = 0; i < nr * nr; ++i) g0[i] = 0.0;
  for (int i = 0; i < nn * nn; ++i) {
    g1[i] = 0.0;
    g2[i] = 0.0;
  }
  for (int i = 0; i < nn * nr; ++i) g3[i] = 0.0;
  // The diagonal loss terms accumulate over ALL regions (also unsolved ones), in
  // the reference's loop order (from-region outer, to-region inner).
  for (int rf = 0; rf < nr; ++rf) {
    const int Rf = r0 + rf;
    for (int Rt = 0; Rt < nreg; ++Rt) {
      if (Rt == Rf) continue;
      const double fx = gm.f_exchange[Rt + 3 * Rf];
      g0[rf + nr * rf] = g0[rf + nr * rf] - tan0 * fx;
      const int rt = Rt - r0;
      if (rt >= 0 && rt < nr) g0[rt + nr * rf] = +tan0 * fx;
      for (int js = 0; js < ns; ++js) {
        const int ifr = js + rf * ns;
        g1[ifr + nn * ifr] = g1[ifr + nn * ifr] - a.lg.tan_ang[js] * fx;
        if (rt >= 0 && rt < nr) g1[(js + rt * ns) + nn * ifr] = +a.lg.tan_ang[js] * fx;
      }
    }
  }
  for (int r = 0; r < nr; ++r) {
    const int Rr = r0 + r;
    if (c.urban)
      g0[r + nr * r] = g0[r + nr * r] - ext[Rr] / zcos - tan0 * gm.f_wall[Rr] * wall_ext;
    else
      g0[r + nr * r] = g0[r + nr * r] - ext[Rr] / cos_sza;
    for (int js = 0; js < ns; ++js) {
      const int i = js + r * ns;
      if (c.urban)
        g1[i + nn * i] = g1[i + nn * i] - ext[Rr] / a.lg.mu[js] - a.lg.tan_ang[js] * gm.f_wall[Rr] * wall_ext;
      else
        g1[i + nn * i] = g1[i + nn * i] - ext[Rr] / a.lg.mu[js];
    }
  }
  for (int jf = 0; jf < ns; ++jf)
    for (int jt = 0; jt < ns; ++jt)
      for (int r = 0; r < nr; ++r) {
        const int Rr = r0 + r;
        const int ifr = jf + r * ns, ito = jt + r * ns;
        if (c.urban)
          g2[ito + nn * ifr] = 0.5 * (a.lg.weight[jt] * ext[Rr] * ssa[Rr] / a.lg.mu[jf] +
                                      a.lg.vweight[jt] * a.lg.tan_ang[jf] * gm.f_wall[Rr] * wall_factor);
        else
          g2[ito + nn * ifr] = 0.5 * a.lg.weight[jt] * ext[Rr] * ssa[Rr] / a.lg.mu[jf];
      }
  for (int i = 0; i < nn * nn; ++i) g1[i] = g1[i] + g2[i];
  for (int r = 0; r < nr; ++r)
    for (int js = 0; js < ns; ++js) {
      const int Rr = r0 + r;
      if (c.urban)
        g3[(js + r * ns) + nn * r] =
            0.5 * (a.lg.weight[js] * ext[Rr] * ssa[Rr] + a.lg.vweight[js] * sin0 * gm.f_wall[Rr] * wall_factor);
      else
        g3[(js + r * ns) + nn * r] = 0.5 * a.lg.weight[js] * ext[Rr] * ssa[Rr];
    }

  double R[NC * NC], T[NC * NC], Idiff[NC * NC], Sup[NC * 3], Sdn[NC * 3], Idd[NC * 3], E[9], Idir[9];
  RadtoolWork<NC> w;
  for (int r = 0; r < nr; ++r) {
    w.frac[r] = gm.frac[r0 + r];
    for (int js = 0; js < ns; ++js) w.ninv[js + r * ns] = a.lg.weight[js] * a.lg.mu[js] * gm.frac[r0 + r];
  }
  const int nfail = calc_matrices_sw<NC>(nn, nr, a.cp.dz[il], g0, g1, g2, g3, R, T, Sup, Sdn, E, Idir, Idiff,
                                         Idd, w);
  count_failure(a.status, nfail);

  // scatter into full-size (n x n etc.) scratch matrices, zero outside the solved block
  const int d = nreg, nlev = a.lmax, i0 = r0 * ns;
  double *S = a.layer;
  int e = 0;
  auto put_nn = [&](const double *M) {
    for (int j = 0; j < n; ++j)
      for (int i = 0; i < n; ++i) {
        const int bi = i - i0, bj = j - i0;
        const bool in = bi >= 0 && bi < nn && bj >= 0 && bj < nn;
        S[sidx(e + i + n * j, lev, nlev, width, q)] = in ? M[bi + nn * bj] : 0.0;
      }
    e += n * n;
  };
  auto put_nd = [&](const double *M) {
    for (int j = 0; j < d; ++j)
      for (int i = 0; i < n; ++i) {
        const int bi = i - i0, bj = j - r0;
        const bool in = bi >= 0 && bi < nn && bj >= 0 && bj < nr;
        S[sidx(e + i + n * j, lev, nlev, width, q)] = in ? M[bi + nn * bj] : 0.0;
      }
    e += n * d;
  };
  auto put_dd = [&](const double *M) {
    for (int j = 0; j < d; ++j)
      for (int i = 0; i < d; ++i) {
        const int bi = i - r0, bj = j - r0;
        const bool in = bi >= 0 && bi < nr && bj >= 0 && bj < nr;
        S[sidx(e + i + d * j, lev, nlev, width, q)] = in ? M[bi + nr * bj] : 0.0;
      }
    e += d * d;
  };
  put_nn(R);
  put_nn(T);
  put_nn(Idiff);
  put_nd(Sup);
  put_nd(Sdn);
  put_nd(Idd);
  put_dd(E);
  put_dd(Idir);
}

template <int NS>
SSB_HD inline void layer_problem_lw(const ClassArgs &a, int q, int lev) {
  constexpr int NC = 3 * NS;
  const SolveCfg &c = a.cfg;
  const int nspec = c.nspec, nreg = c.nreg, ns = c.ns, n = nreg * ns;
  const int ic = q / nspec, g = q % nspec;
  const int col = a.cols[ic];
  if (lev >= a.nlay[col]) return;
  const int il = a.istartlay[col] - 1 + lev;
  const int width = a.ne_layer;  // element count of the layer scratch (sidx)
  const double bf = c.urban ? a.cp.building_fraction[il] : 0.0;
  const double bs = c.urban ? a.cp.building_scale[il] : 0.0;
  const bool veg = nreg > 1 || !c.urban;
  const double vf = (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il] : 0.0;
  const double vs = (veg && a.cp.veg_scale) ? a.cp.veg_scale[il] : 1.0;
  const double ve = (veg && a.cp.veg_ext) ? a.cp.veg_ext[il] : 0.0;
  const double vcf = (c.urban && nreg > 1 && a.cp.veg_contact_fraction) ? a.cp.veg_contact_fraction[il] : 0.0;
  const double vfsd = (nreg == 3) ? a.cp.veg_fsd[il] : 0.0;
  LayerGeom gm;
  layer_geometry(c, bf, bs, vf, vs, vcf, vfsd, a.lg.vadjustment2, gm);

  double ext[3], ssa[3], planck[3];
  ext[0] = SSB_LAY(a.lw.air_ext, g, il);
  ssa[0] = SSB_LAY(a.lw.air_ssa, g, il);
  planck[0] = SSB_LAY(a.lw.clear_air_planck, g, il);
  double vssa = 0.0, vplanck = 0.0, vaplanck = 0.0;
  if (nreg > 1) {
    vssa = SSB_LAY(a.lw.veg_ssa, g, il);
    vplanck = SSB_LAY(a.lw.veg_planck, g, il);
    vaplanck = SSB_LAY(a.lw.veg_air_planck, g, il);
  }
  for (int r = 1; r < nreg; ++r) {
    if (nreg == 2) {
      ext[r] = ext[0] + ve;
      ssa[r] = (ext[0] * ssa[0] + ve * vssa) / dmax(ext[r], 1.0e-8);
      planck[r] = (ext[0] * (1.0 - ssa[0]) * vaplanck + ve * (1.0 - vssa) * vplanck) /
                  dmax(ext[r] * (1.0 - ssa[r]), 1.0e-8);
    } else {
      const double od = gm.od_scaling[r];
      ext[r] = ext[0] + od * ve;
      ssa[r] = (ext[0] * ssa[0] + od * ve * vssa) / dmax(ext[r], 1.0e-8);
      planck[r] = (ext[0] * (1.0 - ssa[0]) * vaplanck + od * ve * (1.0 - vssa) * vplanck) /
                  dmax(ext[r] * (1.0 - ssa[r]), 1.0e-8);
    }
  }
  const double wall_ext = 1.0;
  // the reference reads spectral index 1 for every interval here (urban_lw:392)
  const double wall_factor = c.urban ? 1.0 - SSB_LAY(a.lw.wall_emissivity, 0, il) : 0.0;

  const int r0 = gm.r0, nr = gm.nr, nn = nr * ns;
  double g1[NC * NC], g2[NC * NC], brate[NC];
  for (int i = 0; i < nn * nn; ++i) {
    g1[i] = 0.0;
    g2[i] = 0.0;
  }
  for (int rf = 0; rf < nr; ++rf) {
    const int Rf = r0 + rf;
    for (int Rt = 0; Rt < nreg; ++Rt) {
      if (Rt == Rf) continue;
      const double fx = gm.f_exchange[Rt + 3 * Rf];
      const int rt = Rt - r0;
      for (int js = 0; js < ns; ++js) {
        const int ifr = js + rf * ns;
        g1[ifr + nn * ifr] = g1[ifr + nn * ifr] - a.lg.tan_ang[js] * fx;
        if (rt >= 0 && rt < nr) g1[(js + rt * ns) + nn * ifr] = +a.lg.tan_ang[js] * fx;
      }
    }
  }
  for (int r = 0; r < nr; ++r) {
    const int Rr = r0 + r;
    for (int js = 0; js < ns; ++js) {
      const int i = js + r * ns;
      if (c.urban)
        g1[i + nn * i] = g1[i + nn * i] - ext[Rr] / a.lg.mu[js] - a.lg.tan_ang[js] * gm.f_wall[Rr] * wall_ext;
      else
        g1[i + nn * i] = g1[i + nn * i] - ext[Rr] / a.lg.mu[js];
    }
  }
  for (int jf = 0; jf < ns; ++jf)
    for (int jt = 0; jt < ns; ++jt)
      for (int r = 0; r < nr; ++r) {
        const int Rr = r0 + r;
        const int ifr = jf + r * ns, ito = jt + r * ns;
        if (c.urban)
          g2[ito + nn * ifr] = 0.5 * (a.lg.weight[jt] * ext[Rr] * ssa[Rr] / a.lg.mu[jf] +
                                      a.lg.vweight[jt] * a.lg.tan_ang[jf] * gm.f_wall[Rr] * wall_factor);
        else
          g2[ito + nn * ifr] = (0.5 * a.lg.weight[jt] / a.lg.mu[jf]) * ext[Rr] * ssa[Rr];
      }
  for (int i = 0; i < nn * nn; ++i) g1[i] = g1[i] + g2[i];

  // emission rates and the bookkeeping terms of urban_lw:447-476 (all regions)
  double emiss_factor = 0.0;
  for (int js = 0; js < ns; ++js) emiss_factor += a.lg.hweight[js] / a.lg.mu[js];
  emiss_factor = 2.0 * emiss_factor;
  const int d = nreg, nlev = a.lmax;
  double *S = a.layer;
  const int e_book = 3 * n * n + 2 * n;  // emiss_reg[nreg], emiss_air[nreg], emiss_veg[nreg], emiss_wall
  const double wall_emission = c.urban ? SSB_LAY(a.lw.wall_emission, g, il) : 0.0;
  for (int Rr = 0; Rr < nreg; ++Rr) {
    const double volume_emiss = gm.frac[Rr] * (ext[Rr] * (1.0 - ssa[Rr]) * planck[Rr]);
    const double wall_emiss = c.urban ? gm.norm_perim_wall[Rr] * a.lg.vadjustment * wall_emission : 0.0;
    const int r = Rr - r0;
    if (r >= 0 && r < nr)
      for (int js = 0; js < ns; ++js) {
        if (c.urban)
          brate[js + r * ns] = (a.lg.hweight[js] / a.lg.mu[js]) * volume_emiss + (0.5 * a.lg.vweight[js]) * wall_emiss;
        else
          brate[js + r * ns] = (a.lg.hweight[js] / a.lg.mu[js]) * volume_emiss;
      }
    S[sidx(e_book + Rr, lev, nlev, width, q)] = emiss_factor * volume_emiss;
    double e_air = 0.0, e_veg = 0.0;
    if (Rr > 0) {
      e_air = emiss_factor * gm.frac[Rr] * ext[0] * (1.0 - ssa[0]) * vaplanck;
      e_veg = emiss_factor * gm.frac[Rr] * ve * (1.0 - vssa) * vplanck * gm.od_scaling[Rr];
    }
    S[sidx(e_book + d + Rr, lev, nlev, width, q)] = e_air;
    S[sidx(e_book + 2 * d + Rr, lev, nlev, width, q)] = e_veg;
  }
  {
    double s = 0.0;
    for (int Rr = 0; Rr < nreg; ++Rr) s += gm.norm_perim_wall[Rr];
    S[sidx(e_book + 3 * d, lev, nlev, width, q)] = c.urban ? (s * a.lg.vadjustment) * wall_emission : 0.0;
  }

  double R[NC * NC], T[NC * NC], IF[NC * NC], src[NC], isrc[NC];
  RadtoolWork<NC> w;
  for (int r = 0; r < nr; ++r) {
    w.frac[r] = gm.frac[r0 + r];
    for (int js = 0; js < ns; ++js) w.ninv[js + r * ns] = a.lg.weight[js] * a.lg.mu[js] * gm.frac[r0 + r];
  }
  const int nfail = calc_matrices_lw<NC>(nn, a.cp.dz[il], g1, g2, brate, R, T, src, IF, isrc, w);
  count_failure(a.status, nfail);

  const int i0 = r0 * ns;
  int e = 0;
  auto put_nn = [&](const double *M) {
    for (int j = 0; j < n; ++j)
      for (int i = 0; i < n; ++i) {
        const int bi = i - i0, bj = j - i0;
        const bool in = bi >= 0 && bi < nn && bj >= 0 && bj < nn;
        S[sidx(e + i + n * j, lev, nlev, width, q)] = in ? M[bi + nn * bj] : 0.0;
      }
    e += n * n;
  };
  auto put_n = [&](const double *v) {
    for (int i = 0; i < n; ++i) {
      const int bi = i - i0;
      S[sidx(e + i, lev, nlev, width, q)] = (bi >= 0 && bi < nn) ? v[bi] : 0.0;
    }
    e += n;
  };
  put_nn(R);
  put_nn(T);
  put_nn(IF);
  put_n(src);
  put_n(isrc);
}

// ---------------------------------------------------------------------------
// Small helpers for the sweeps
// ---------------------------------------------------------------------------
struct ScratchIO {
  double *base;
  int nlev, nelem, q;
  SSB_HDI void load(int e0, int cnt, int lev, double *dst) const {
    for (int i = 0; i < cnt; ++i) dst[i] = base[sidx(e0 + i, lev, nlev, nelem, q)];
  }
  SSB_HDI void store(int e0, int cnt, int lev, const double *src) const {
    for (int i = 0; i < cnt; ++i) base[sidx(e0 + i, lev, nlev, nelem, q)] = src[i];
  }
};

// C (nu*s x p) = (U (x) I_s) B, U is nu x nl at [up + nu*lo], B is (nl*s x p); zero entries skipped
SSB_HDI void expand_left(int nu, int nl, int s, int p, const double *U, const double *B, double *C) {
  const int rc = nu * s, rb = nl * s;
  for (int i = 0; i < rc * p; ++i) C[i] = 0.0;
  for (int up = 0; up < nu; ++up)
    for (int lo = 0; lo < nl; ++lo) {
      const double u = U[up + nu * lo];
      if (u != 0.0)
        for (int j = 0; j < p; ++j)
          for (int js = 0; js < s; ++js)
            C[(up * s + js) + rc * j] = C[(up * s + js) + rc * j] + u * B[(lo * s + js) + rb * j];
    }
}
// C (p x nu*s) = A (V (x) I_s), V is nl x nu at [lo + nl*up], A is (p x nl*s)
SSB_HDI void expand_right(int nl, int nu, int s, int p, const double *A, const double *V, double *C) {
  for (int i = 0; i < p * nu * s; ++i) C[i] = 0.0;
  for (int up = 0; up < nu; ++up)
    for (int lo = 0; lo < nl; ++lo) {
      const double v = V[lo + nl * up];
      if (v != 0.0)
        for (int i = 0; i < p; ++i)
          for (int js = 0; js < s; ++js)
            C[i + p * (up * s + js)] = C[i + p * (up * s + js)] + A[i + p * (lo * s + js)] * v;
    }
}
// y (nt*s) = (M (x) I_s) x, M is nt x nf at [to + nt*from]
SSB_HDI void expand_vec(int nt, int nf, int s, const double *M, const double *x, double *y) {
  for (int i = 0; i < nt * s; ++i) y[i] = 0.0;
  for (int to = 0; to < nt; ++to)
    for (int fr = 0; fr < nf; ++fr) {
      const double m = M[to + nt * fr];
      if (m != 0.0)
        for (int js = 0; js < s; ++js) y[to * s + js] = y[to * s + js] + m * x[fr * s + js];
    }
}

SSB_HDI double vsum(const double *v, int i0, int cnt) {
  double s = 0.0;
  for (int i = i0; i < i0 + cnt; ++i) s += v[i];
  return s;
}

// zero every allocated member of one (column, interval) slice (canopy_flux%zero,
// radsurf_canopy_flux.F90:286-341); the non-spectral members are zeroed by the
// thread that owns them (`own_scalars`).
SSB_HD inline void zero_column(const ssb200_canopy_flux &f, int nspec, int g, int col, int il1, int nlay,
                               bool own_scalars, int ls = 1) {
  auto zc = [&](double *p) {
    if (p) p[(size_t)g + (size_t)nspec * col] = 0.0;
  };
  auto zl = [&](double *p) {
    if (p)
      for (int l = 0; l < nlay; ++l) p[(size_t)g + (size_t)nspec * (il1 + l * ls)] = 0.0;
  };
  zc(f.ground_dn);
  zc(f.ground_net);
  zc(f.ground_vertical_diff);
  zc(f.top_dn);
  zc(f.top_net);
  zc(f.ground_dn_dir);
  zc(f.top_dn_dir);
  zl(f.roof_in);
  zl(f.roof_net);
  zl(f.wall_in);
  zl(f.wall_net);
  zl(f.roof_in_dir);
  zl(f.wall_in_dir);
  zl(f.clear_air_abs);
  zl(f.veg_abs);
  zl(f.veg_air_abs);
  zl(f.veg_abs_dir);
  zl(f.flux_dn_layer_top);
  zl(f.flux_up_layer_top);
  zl(f.flux_dn_layer_base);
  zl(f.flux_up_layer_base);
  zl(f.flux_dn_dir_layer_top);
  zl(f.flux_dn_dir_layer_base);
  if (own_scalars) {
    if (f.ground_sunlit_frac) f.ground_sunlit_frac[col] = 0.0;
    for (int l = 0; l < nlay; ++l) {
      if (f.roof_sunlit_frac) f.roof_sunlit_frac[il1 + l * ls] = 0.0;
      if (f.wall_sunlit_frac) f.wall_sunlit_frac[il1 + l * ls] = 0.0;
      if (f.veg_sunlit_frac) f.veg_sunlit_frac[il1 + l * ls] = 0.0;
    }
  }
}

#define SSB_FC(f, member) (f.member[(size_t)g + (size_t)nspec * col])
#define SSB_FL(f, member, il) (f.member[(size_t)g + (size_t)nspec * (il)])

// read the geometry inputs of layer `il` and evaluate the layer geometry
SSB_HD inline void geometry_of_layer(const ClassArgs &a, int il, double wall_adj, LayerGeom &gm, double &bf,
                                     double &vf, double &ve) {
  const SolveCfg &c = a.cfg;
  const bool veg = c.nreg > 1 || !c.urban;
  bf = c.urban ? a.cp.building_fraction[il] : 0.0;
  const double bs = c.urban ? a.cp.building_scale[il] : 0.0;
  vf = (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il] : 0.0;
  const double vs = (veg && a.cp.veg_scale) ? a.cp.veg_scale[il] : 1.0;
  ve = (veg && a.cp.veg_ext) ? a.cp.veg_ext[il] : 0.0;
  const double vcf = (c.urban && c.nreg > 1 && a.cp.veg_contact_fraction) ? a.cp.veg_contact_fraction[il] : 0.0;
  const double vfsd = (c.nreg == 3) ? a.cp.veg_fsd[il] : 0.0;
  layer_geometry(c, bf, bs, vf, vs, vcf, vfsd, wall_adj, gm);
}

// U, V at interface k of the column starting at packed layer il1
SSB_HD inline void overlap_at(const ClassArgs &a, int il1, int nlay, int k, double *U, double *V) {
  const SolveCfg &c = a.cfg;
  double fb[3] = {0, 0, 0}, fa[3] = {0, 0, 0}, fu[3], fl[4];
  const bool veg = c.nreg > 1 || !c.urban;
  if (k >= 1) {
    const int il = il1 + k - 1;
    region_fractions(c, c.urban ? a.cp.building_fraction[il] : 0.0,
                     (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il] : 0.0, fb);
  }
  if (k < nlay) {
    const int il = il1 + k;
    region_fractions(c, c.urban ? a.cp.building_fraction[il] : 0.0,
                     (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il] : 0.0, fa);
  }
  interface_fractions(c, k, nlay, fb, fa, fu, fl);
  overlap_interface(c, fu, fl, U, V);
}

// ---------------------------------------------------------------------------
// Column sweeps, shortwave
// ---------------------------------------------------------------------------
template <int NS>
SSB_HD inline void column_sweeps_sw(const ClassArgs &a, int q) {
  constexpr int NC = 3 * NS, MC = 4 * NS;
  const SolveCfg &c = a.cfg;
  const int nspec = c.nspec, nreg = c.nreg, ns = c.ns, n = nreg * ns, d = nreg;
  const int nrb = c.urban ? nreg + 1 : nreg, m = nrb * ns, db = nrb;
  const int ic = q / nspec, g = q % nspec;
  const int col = a.cols[ic];
  const int nlay = a.nlay[col], il1 = a.istartlay[col] - 1;
  const ssb200_canopy_flux &fdir = a.f1, &fdif = a.f2;
  const double cos_sza = a.cp.cos_sza[col];

  // most transparent interval (urban_sw:310): first minimum of the column optical depth
  int itransp = 0;
  if (nspec > 1) {
    double best = 0.0;
    for (int gg = 0; gg < nspec; ++gg) {
      double od = 0.0;
      for (int l = 0; l < nlay; ++l) od += a.sw.air_ext[(size_t)gg + (size_t)nspec * (il1 + l)] * a.cp.dz[il1 + l];
      if (gg == 0 || od < best) {
        best = od;
        itransp = gg;
      }
    }
  }
  const bool own = (g == itransp);
  zero_column(fdir, nspec, g, col, il1, nlay, own);
  zero_column(fdif, nspec, g, col, il1, nlay, own);
  if (!(cos_sza > 0.0)) return;  // night: fluxes zero, bc_out untouched (radsurf_interface.F90:258-260)

  const double zcos = c.urban ? dmax(cos_sza, 1.0e-6) : cos_sza;
  const double sin0 = c.urban ? sqrt(1.0 - zcos * zcos) : 0.0;
  const double galb = a.sw.ground_albedo[(size_t)g + (size_t)nspec * col];
  const double galb_dir = (a.use_sw_direct_albedo ? a.sw.ground_albedo_dir : a.sw.ground_albedo)[(size_t)g + (size_t)nspec * col];

  const ScratchIO L{a.layer, a.lmax, a.ne_layer, q};
  const ScratchIO W{a.sweep, a.lmax + 1, a.ne_sweep, q};
  // layer scratch offsets
  const int oR = 0, oT = n * n, oIdiff = 2 * n * n, oSup = 3 * n * n, oSdn = oSup + n * d, oIdd = oSdn + n * d,
            oE = oIdd + n * d, oIdir = oE + d * d;
  // sweep scratch offsets
  const int oAa = 0, oDa = n * n, oDen = oDa + n * d, oAb = oDen + n * n, oDb = oAb + m * m, oU = oDb + m * db,
            oV = oU + nreg * nrb;

  double Aa[NC * NC], Da[NC * 3], R[NC * NC], T[NC * NC], t1[NC * NC], t2[NC * NC], lu[NC * NC];
  double Ab[MC * MC], Db[MC * 4], tA[MC * MC];
  double Su[NC * 3], Sd[NC * 3], E[9], U[12], V[12];

  // -- Section 4: albedo of the scene below each interface -------------------
  for (int i = 0; i < n * n; ++i) Aa[i] = 0.0;
  for (int i = 0; i < n * d; ++i) Da[i] = 0.0;
  for (int r = 0; r < nreg; ++r)
    for (int jt = 0; jt < ns; ++jt) {
      Da[(jt + r * ns) + n * r] = zcos * galb_dir * a.lg.hweight[jt];
      for (int jf = 0; jf < ns; ++jf) Aa[(jt + r * ns) + n * (jf + r * ns)] = galb * a.lg.hweight[jt];
    }
  W.store(oAa, n * n, 0, Aa);
  W.store(oDa, n * d, 0, Da);
  for (int jl = 0; jl < nlay; ++jl) {
    const int il = il1 + jl;
    L.load(oR, n * n, jl, R);
    L.load(oT, n * n, jl, T);
    L.load(oSup, n * d, jl, Su);
    L.load(oSdn, n * d, jl, Sd);
    L.load(oE, d * d, jl, E);
    // denominator = I - Aa R
    mat_mul(n, n, n, Aa, R, t1);
    for (int i = 0; i < n * n; ++i) t1[i] = -t1[i];
    for (int i = 0; i < n; ++i) t1[i + n * i] = 1.0 + t1[i + n * i];
    W.store(oDen, n * n, jl, t1);
    // a_below = R + T D^-1 (Aa T)
    mat_mul(n, n, n, Aa, T, t2);
    double *X = tA;  // n x n
    solve_mat(n, t1, t2, X, lu);
    mat_mul(n, n, n, T, X, t2);
    for (int i = 0; i < m * m; ++i) Ab[i] = 0.0;
    for (int j = 0; j < n; ++j)
      for (int i = 0; i < n; ++i) Ab[i + m * j] = R[i + n * j] + t2[i + n * j];
    // d_below = Sup + T D^-1 (Da E + Aa Sdn)
    double r1[NC * 3], r2[NC * 3];
    mat_mul(n, d, d, Da, E, r1);
    mat_mul(n, n, d, Aa, Sd, r2);
    for (int i = 0; i < n * d; ++i) r1[i] = r1[i] + r2[i];
    for (int i = 0; i < n * n; ++i) lu[i] = t1[i];
    solve_rect(n, d, lu, r1, r2);
    mat_mul(n, n, d, T, r2, r1);
    for (int i = 0; i < m * db; ++i) Db[i] = 0.0;
    for (int j = 0; j < d; ++j)
      for (int i = 0; i < n; ++i) Db[i + m * j] = Su[i + n * j] + r1[i + n * j];
    if (c.urban) {
      const double ralb = SSB_LAY(a.sw.roof_albedo, g, il);
      const double ralb_dir = a.sw.roof_albedo_dir ? SSB_LAY(a.sw.roof_albedo_dir, g, il) : ralb;
      for (int js = 0; js < ns; ++js) {
        for (int j2 = 0; j2 < ns; ++j2) Ab[(n + js) + m * (n + j2)] = ralb * a.lg.hweight[js];
        Db[(n + js) + m * nreg] = zcos * ralb_dir * a.lg.hweight[js];
      }
    }
    overlap_at(a, il1, nlay, jl + 1, U, V);
    // a_above(next) = (U (x) I)(a_below (V (x) I)) ; d_above(next) = (U (x) I)(d_below V)
    expand_right(nrb, nreg, ns, m, Ab, V, tA);  // m x n
    expand_left(nreg, nrb, ns, n, U, tA, Aa);   // n x n
    double dv[MC * 3];
    mat_mul(m, db, d, Db, V, dv);  // V is (nrb x nreg) = (db x d)
    expand_left(nreg, nrb, ns, d, U, dv, Da);
    W.store(oAb, m * m, jl + 1, Ab);
    W.store(oDb, m * db, jl + 1, Db);
    W.store(oU, nreg * nrb, jl + 1, U);
    W.store(oV, nreg * nrb, jl + 1, V);
    W.store(oAa, n * n, jl + 1, Aa);
    W.store(oDa, n * d, jl + 1, Da);
  }
  // top-of-canopy boundary conditions (urban_sw:672-674)
  double talb_diff = 0.0, talb_dir = 0.0;
  {
    for (int i = 0; i < ns; ++i) {
      double s = 0.0;
      for (int j = 0; j < ns; ++j) s = s + Aa[i + n * j] * a.lg.hweight[j];
      talb_diff += s;
    }
    double s = 0.0;
    for (int js = 0; js < ns; ++js) s += Da[js];
    talb_dir = s / zcos;
    a.bc.sw_albedo[(size_t)g + (size_t)nspec * col] = talb_diff;
    a.bc.sw_albedo_dir[(size_t)g + (size_t)nspec * col] = talb_dir;
  }

  // -- Section 5: two downward passes ----------------------------------------
  double dir_above[3], dir_below[4], diff_above[NC], diff_below[MC], up_above[NC], up_below[MC];
  double refl[NC], rhs[NC], tmpv[NC], conv[NC], iflux_dir[3], iflux_diff[NC], ddir[3];
  for (int pass = 0; pass < 2; ++pass) {
    const bool direct = (pass == 0);
    const ssb200_canopy_flux &f = direct ? fdir : fdif;
    for (int i = 0; i < 3; ++i) dir_above[i] = 0.0;
    for (int i = 0; i < n; ++i) diff_above[i] = 0.0;
    for (int i = 0; i < n; ++i) up_above[i] = 0.0;
    double flux_dn_dir_clear = 1.0 / zcos;
    if (direct) {
      dir_above[0] = 1.0 / zcos;
      SSB_FC(f, top_dn_dir) = 1.0;
      SSB_FC(f, top_dn) = 1.0;
      SSB_FC(f, top_net) = 1.0 * (1.0 - talb_dir);
      if (c.urban && own && f.roof_sunlit_frac && nlay > 0) f.roof_sunlit_frac[il1 + nlay - 1] = 1.0;
    } else {
      for (int js = 0; js < ns; ++js) diff_above[js] = a.lg.hweight[js];
      SSB_FC(f, top_dn_dir) = 0.0;
      SSB_FC(f, top_dn) = 1.0;
      SSB_FC(f, top_net) = 1.0 - talb_diff;
    }
    for (int jl = nlay - 1; jl >= 0; --jl) {
      const int il = il1 + jl;
      LayerGeom gm;
      double bf, vf, ve;
      geometry_of_layer(a, il, 1.0, gm, bf, vf, ve);
      W.load(oV, nreg * nrb, jl + 1, V);
      W.load(oAb, m * m, jl + 1, Ab);
      expand_vec(nrb, nreg, ns, V, diff_above, diff_below);
      mat_vec(m, m, Ab, diff_below, up_below);
      if (direct) {
        W.load(oDb, m * db, jl + 1, Db);
        mat_vec(nrb, nreg, V, dir_above, dir_below);
        double t[MC];
        mat_vec(m, db, Db, dir_below, t);
        for (int i = 0; i < m; ++i) up_below[i] = up_below[i] + t[i];
      }
      if (c.urban) {
        if (direct) {
          SSB_FL(f, roof_in_dir, il) = zcos * dir_below[nreg];
          SSB_FL(f, roof_in, il) = SSB_FL(f, roof_in_dir, il) + vsum(diff_below, n, ns);
        } else {
          SSB_FL(f, roof_in, il) = +vsum(diff_below, n, ns);
        }
        SSB_FL(f, roof_net, il) = SSB_FL(f, roof_in, il) - vsum(up_below, n, ns);
      }
      W.load(oAa, n * n, jl, Aa);
      W.load(oDen, n * n, jl, t1);
      L.load(oT, n * n, jl, T);
      mat_vec(n, n, T, diff_below, rhs);
      if (direct) {
        L.load(oE, d * d, jl, E);
        W.load(oDa, n * d, jl, Da);
        L.load(oR, n * n, jl, R);
        L.load(oSdn, n * d, jl, Sd);
        double da_new[3];
        mat_vec(d, d, E, dir_below, da_new);
        for (int i = 0; i < d; ++i) ddir[i] = dir_below[i] - da_new[i];
        for (int i = 0; i < d; ++i) dir_above[i] = da_new[i];
        mat_vec(n, d, Da, dir_above, refl);
        mat_vec(n, n, R, refl, tmpv);
        for (int i = 0; i < n; ++i) rhs[i] = rhs[i] + tmpv[i];
        mat_vec(n, d, Sd, dir_below, tmpv);
        for (int i = 0; i < n; ++i) rhs[i] = rhs[i] + tmpv[i];
      }
      solve_vec(n, t1, rhs, diff_above, lu);
      mat_vec(n, n, Aa, diff_above, up_above);
      if (direct)
        for (int i = 0; i < n; ++i) up_above[i] = up_above[i] + refl[i];

      if (f.flux_dn_layer_top) {
        if (direct) {
          SSB_FL(f, flux_dn_dir_layer_top, il) = zcos * vsum(dir_below, 0, nreg);
          SSB_FL(f, flux_dn_layer_top, il) = SSB_FL(f, flux_dn_dir_layer_top, il) + vsum(diff_below, 0, n);
          SSB_FL(f, flux_dn_dir_layer_base, il) = zcos * vsum(dir_above, 0, nreg);
          SSB_FL(f, flux_dn_layer_base, il) = SSB_FL(f, flux_dn_dir_layer_base, il) + vsum(diff_above, 0, n);
        } else {
          SSB_FL(f, flux_dn_layer_top, il) = vsum(diff_below, 0, n);
          SSB_FL(f, flux_dn_layer_base, il) = vsum(diff_above, 0, n);
        }
        SSB_FL(f, flux_up_layer_top, il) = vsum(up_below, 0, n);
        SSB_FL(f, flux_up_layer_base, il) = vsum(up_above, 0, n);
      }

      // integrated fluxes across the layer
      for (int i = 0; i < n; ++i) conv[i] = diff_below[i] - diff_above[i] - up_below[i] + up_above[i];
      L.load(oIdiff, n * n, jl, R);  // R buffer reused
      mat_vec(n, n, R, conv, iflux_diff);
      for (int i = 0; i < 3; ++i) iflux_dir[i] = 0.0;
      if (direct) {
        double Idir[9];
        L.load(oIdir, d * d, jl, Idir);
        mat_vec(d, d, Idir, ddir, iflux_dir);
        L.load(oIdd, n * d, jl, Su);  // Su buffer reused
        mat_vec(n, d, Su, ddir, tmpv);
        for (int i = 0; i < n; ++i) iflux_diff[i] = iflux_diff[i] + tmpv[i];
      }
      auto sum_over_mu = [&](int r) {
        double s = 0.0;
        for (int js = 0; js < ns; ++js) s += iflux_diff[r * ns + js] * (1.0 / a.lg.mu[js]);
        return s;
      };
      auto sum_tan = [&](int r) {
        double s = 0.0;
        for (int js = 0; js < ns; ++js) s += iflux_diff[r * ns + js] * a.lg.tan_ang[js];
        return s;
      };
      const double air_ext = SSB_LAY(a.sw.air_ext, g, il);
      const double air_abs = air_ext * (1.0 - SSB_LAY(a.sw.air_ssa, g, il));
      if (direct)
        SSB_FL(f, clear_air_abs, il) = SSB_FL(f, clear_air_abs, il) + air_abs * (iflux_dir[0] + sum_over_mu(0));
      else
        SSB_FL(f, clear_air_abs, il) = SSB_FL(f, clear_air_abs, il) + air_abs * sum_over_mu(0);
      if (nreg > 1) {
        const double vabs = ve * (1.0 - SSB_LAY(a.sw.veg_ssa, g, il));
        for (int r = 1; r < nreg; ++r) {
          if (direct) {
            SSB_FL(f, veg_air_abs, il) = SSB_FL(f, veg_air_abs, il) + air_abs * (iflux_dir[r] + sum_over_mu(r));
            SSB_FL(f, veg_abs_dir, il) = SSB_FL(f, veg_abs_dir, il) + vabs * iflux_dir[r] * gm.od_scaling[r];
            SSB_FL(f, veg_abs, il) =
                SSB_FL(f, veg_abs, il) + vabs * (iflux_dir[r] + sum_over_mu(r)) * gm.od_scaling[r];
          } else {
            SSB_FL(f, veg_air_abs, il) = SSB_FL(f, veg_air_abs, il) + air_abs * sum_over_mu(r);
            SSB_FL(f, veg_abs, il) = SSB_FL(f, veg_abs, il) + vabs * sum_over_mu(r) * gm.od_scaling[r];
          }
        }
      }
      if (c.urban) {
        const double walb = SSB_LAY(a.sw.wall_albedo, g, il);
        if (direct) {
          for (int r = 0; r < nreg; ++r)
            SSB_FL(f, wall_in_dir, il) = SSB_FL(f, wall_in_dir, il) + gm.f_wall[r] * sin0 * iflux_dir[r];
          SSB_FL(f, wall_in, il) = SSB_FL(f, wall_in_dir, il);
        }
        for (int r = 0; r < nreg; ++r) SSB_FL(f, wall_in, il) = SSB_FL(f, wall_in, il) + gm.f_wall[r] * sum_tan(r);
        SSB_FL(f, wall_net, il) = SSB_FL(f, wall_in, il) * (1.0 - walb);
      }
      if (direct) {
        // spectrally independent sunlit fractions from the most transparent interval
        // (urban_sw:805-848); only the owning thread holds the right interval
        const double nonb_here = c.urban ? 1.0 - bf : 1.0;
        double nonb_above = 1.0;
        if (c.urban && jl + 1 < nlay) nonb_above = 1.0 - a.cp.building_fraction[il + 1];
        if (c.urban) {
          double roof_fraction;
          if (jl == nlay - 1)
            roof_fraction = bf;
          else
            roof_fraction = dmax(0.0, bf - a.cp.building_fraction[il + 1]);
          if (own && f.roof_sunlit_frac)
            f.roof_sunlit_frac[il] = SSB_FL(f, roof_in_dir, il) * nonb_above /
                                     (zcos * flux_dn_dir_clear * dmax(c.min_bld, roof_fraction));
          flux_dn_dir_clear = flux_dn_dir_clear * nonb_here / nonb_above;
        }
        const double air_ext_t = a.sw.air_ext[(size_t)itransp + (size_t)nspec * il];
        const double trans_dir_clear = exp(-air_ext_t * a.cp.dz[il] / zcos);
        double int_flux_dir_clear;
        if (air_ext_t > 0.0)
          int_flux_dir_clear = flux_dn_dir_clear * (1.0 - trans_dir_clear) * zcos / air_ext_t;
        else
          int_flux_dir_clear = flux_dn_dir_clear * a.cp.dz[il];
        if (own) {
          if ((c.urban ? nreg > 1 : true) && f.veg_sunlit_frac && a.cp.veg_ext && a.cp.veg_fraction &&
              a.sw.veg_ssa) {
            const double veg_abs_dir_clear = int_flux_dir_clear * ve * (1.0 - SSB_LAY(a.sw.veg_ssa, g, il)) * vf;
            f.veg_sunlit_frac[il] = SSB_FL(f, veg_abs_dir, il) / dmax(SSB_EPS, veg_abs_dir_clear);
          }
          if (c.urban && f.wall_sunlit_frac)
            f.wall_sunlit_frac[il] = 0.5 * SSB_FL(f, wall_in_dir, il) /
                                     dmax(SSB_EPS, (gm.f_wall_dir_clear * sin0 * int_flux_dir_clear));
        }
        flux_dn_dir_clear = flux_dn_dir_clear * trans_dir_clear;
      }
    }
    if (direct) {
      SSB_FC(f, ground_dn_dir) = zcos * vsum(dir_above, 0, nreg);
      SSB_FC(f, ground_dn) = SSB_FC(f, ground_dn_dir) + vsum(diff_above, 0, n);
    } else {
      SSB_FC(f, ground_dn_dir) = 0.0;
      SSB_FC(f, ground_dn) = vsum(diff_above, 0, n);
    }
    SSB_FC(f, ground_net) = SSB_FC(f, ground_dn) - vsum(up_above, 0, n);
    for (int r = 0; r < nreg; ++r)
      for (int js = 0; js < ns; ++js) {
        const int i = js + r * ns;
        SSB_FC(f, ground_vertical_diff) =
            SSB_FC(f, ground_vertical_diff) + (diff_above[i] + up_above[i]) * a.lg.tan_ang[js] / SSB_PI;
      }
    if (direct && own && f.ground_sunlit_frac)
      f.ground_sunlit_frac[col] = SSB_FC(f, ground_dn_dir) / (zcos * flux_dn_dir_clear);
  }
}

// ---------------------------------------------------------------------------
// Column sweeps, longwave
// ---------------------------------------------------------------------------
template <int NS>
SSB_HD inline void column_sweeps_lw(const ClassArgs &a, int q) {
  constexpr int NC = 3 * NS, MC = 4 * NS;
  const SolveCfg &c = a.cfg;
  const int nspec = c.nspec, nreg = c.nreg, ns = c.ns, n = nreg * ns, d = nreg;
  const int nrb = c.urban ? nreg + 1 : nreg, m = nrb * ns;
  const int ic = q / nspec, g = q % nspec;
  const int col = a.cols[ic];
  const int nlay = a.nlay[col], il1 = a.istartlay[col] - 1;
  const ssb200_canopy_flux &fint = a.f1, &fnorm = a.f2;
  zero_column(fint, nspec, g, col, il1, nlay, g == 0);
  zero_column(fnorm, nspec, g, col, il1, nlay, g == 0);

  const ScratchIO L{a.layer, a.lmax, a.ne_layer, q};
  const ScratchIO W{a.sweep, a.lmax + 1, a.ne_sweep, q};
  const int oR = 0, oT = n * n, oIF = 2 * n * n, oSrc = 3 * n * n, oIsrc = oSrc + n, oBook = oIsrc + n;
  const int oAa = 0, oSa = n * n, oDen = oSa + n, oAb = oDen + n * n, oSb = oAb + m * m, oU = oSb + m,
            oV = oU + nreg * nrb;

  double Aa[NC * NC], Sa[NC], R[NC * NC], T[NC * NC], t1[NC * NC], t2[NC * NC], lu[NC * NC];
  double Ab[MC * MC], Sb[MC], tA[MC * MC], src[NC], U[12], V[12];

  const double gemis = a.lw.ground_emissivity[(size_t)g + (size_t)nspec * col];
  const double gemission = a.lw.ground_emission[(size_t)g + (size_t)nspec * col];
  {
    double frac0[3] = {1.0, 0.0, 0.0};
    if (nlay > 0) {
      const bool veg = nreg > 1 || !c.urban;
      region_fractions(c, c.urban ? a.cp.building_fraction[il1] : 0.0,
                       (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il1] : 0.0, frac0);
    }
    for (int i = 0; i < n * n; ++i) Aa[i] = 0.0;
    for (int r = 0; r < nreg; ++r) {
      for (int jt = 0; jt < ns; ++jt)
        for (int jf = 0; jf < ns; ++jf) Aa[(jt + r * ns) + n * (jf + r * ns)] = (1.0 - gemis) * a.lg.hweight[jt];
      for (int js = 0; js < ns; ++js) Sa[js + r * ns] = (a.lg.hweight[js] * frac0[r]) * gemission;
    }
  }
  W.store(oAa, n * n, 0, Aa);
  W.store(oSa, n, 0, Sa);
  for (int jl = 0; jl < nlay; ++jl) {
    const int il = il1 + jl;
    L.load(oR, n * n, jl, R);
    L.load(oT, n * n, jl, T);
    L.load(oSrc, n, jl, src);
    mat_mul(n, n, n, Aa, R, t1);
    for (int i = 0; i < n * n; ++i) t1[i] = -t1[i];
    for (int i = 0; i < n; ++i) t1[i + n * i] = 1.0 + t1[i + n * i];
    W.store(oDen, n * n, jl, t1);
    mat_mul(n, n, n, Aa, T, t2);
    double *X = tA;
    solve_mat(n, t1, t2, X, lu);
    mat_mul(n, n, n, T, X, t2);
    for (int i = 0; i < m * m; ++i) Ab[i] = 0.0;
    for (int j = 0; j < n; ++j)
      for (int i = 0; i < n; ++i) Ab[i + m * j] = R[i + n * j] + t2[i + n * j];
    // source_below = src + T D^-1 (Sa + Aa src)   (urban_lw:583-587)
    double v1[NC], v2[NC];
    mat_vec(n, n, Aa, src, v1);
    for (int i = 0; i < n; ++i) v1[i] = Sa[i] + v1[i];
    solve_vec(n, t1, v1, v2, lu);
    mat_vec(n, n, T, v2, v1);
    for (int i = 0; i < m; ++i) Sb[i] = 0.0;
    for (int i = 0; i < n; ++i) Sb[i] = src[i] + v1[i];
    if (c.urban) {
      const double bfj = a.cp.building_fraction[il];
      double exposed;
      if (jl < nlay - 1)
        exposed = dmax(0.0, bfj - a.cp.building_fraction[il + 1]);
      else
        exposed = bfj;
      const double remis = SSB_LAY(a.lw.roof_emissivity, g, il), remission = SSB_LAY(a.lw.roof_emission, g, il);
      for (int js = 0; js < ns; ++js) {
        for (int j2 = 0; j2 < ns; ++j2) Ab[(n + js) + m * (n + j2)] = (1.0 - remis) * a.lg.hweight[js];
        Sb[n + js] = a.lg.hweight[js] * remission * exposed;
      }
    }
    overlap_at(a, il1, nlay, jl + 1, U, V);
    expand_right(nrb, nreg, ns, m, Ab, V, tA);
    expand_left(nreg, nrb, ns, n, U, tA, Aa);
    expand_vec(nreg, nrb, ns, U, Sb, Sa);
    W.store(oAb, m * m, jl + 1, Ab);
    W.store(oSb, m, jl + 1, Sb);
    W.store(oU, nreg * nrb, jl + 1, U);
    W.store(oV, nreg * nrb, jl + 1, V);
    W.store(oAa, n * n, jl + 1, Aa);
    W.store(oSa, n, jl + 1, Sa);
  }
  double top_emissivity, top_emission;
  {
    double sAll = 0.0;
    for (int i = 0; i < ns; ++i) {
      double s = 0.0;
      for (int j = 0; j < ns; ++j) s = s + Aa[i + n * j] * a.lg.hweight[j];
      sAll += s;
    }
    top_emissivity = 1.0 - sAll;
    top_emission = vsum(Sa, 0, ns);
    a.bc.lw_emissivity[(size_t)g + (size_t)nspec * col] = top_emissivity;
    a.bc.lw_emission[(size_t)g + (size_t)nspec * col] = top_emission;
  }

  double dn_above[NC], dn_below[MC], up_above[NC], up_below[MC], rhs[NC], tmpv[NC], iflux[NC], book[10];
  for (int pass = 0; pass < 2; ++pass) {
    const bool internal = (pass == 0);
    const ssb200_canopy_flux &f = internal ? fint : fnorm;
    for (int i = 0; i < n; ++i) dn_above[i] = 0.0;
    for (int i = 0; i < n; ++i) up_above[i] = 0.0;
    if (internal) {
      SSB_FC(f, top_dn) = 0.0;
      SSB_FC(f, top_net) = -top_emission;
    } else {
      for (int js = 0; js < ns; ++js) dn_above[js] = a.lg.hweight[js];
      SSB_FC(f, top_dn) = 1.0;
      SSB_FC(f, top_net) = top_emissivity;
    }
    for (int jl = nlay - 1; jl >= 0; --jl) {
      const int il = il1 + jl;
      LayerGeom gm;
      double bf, vf, ve;
      geometry_of_layer(a, il, a.lg.vadjustment2, gm, bf, vf, ve);
      W.load(oV, nreg * nrb, jl + 1, V);
      W.load(oAb, m * m, jl + 1, Ab);
      expand_vec(nrb, nreg, ns, V, dn_above, dn_below);
      mat_vec(m, m, Ab, dn_below, up_below);
      if (internal) {
        W.load(oSb, m, jl + 1, Sb);
        for (int i = 0; i < m; ++i) up_below[i] = up_below[i] + Sb[i];
      }
      if (c.urban) {
        SSB_FL(f, roof_in, il) = vsum(dn_below, n, ns);
        SSB_FL(f, roof_net, il) = SSB_FL(f, roof_in, il) - vsum(up_below, n, ns);
      }
      W.load(oAa, n * n, jl, Aa);
      W.load(oDen, n * n, jl, t1);
      L.load(oT, n * n, jl, T);
      mat_vec(n, n, T, dn_below, rhs);
      if (internal) {
        W.load(oSa, n, jl, Sa);
        L.load(oR, n * n, jl, R);
        L.load(oSrc, n, jl, src);
        mat_vec(n, n, R, Sa, tmpv);
        for (int i = 0; i < n; ++i) rhs[i] = (rhs[i] + tmpv[i]) + src[i];
      }
      solve_vec(n, t1, rhs, dn_above, lu);
      mat_vec(n, n, Aa, dn_above, up_above);
      if (internal)
        for (int i = 0; i < n; ++i) up_above[i] = up_above[i] + Sa[i];
      if (f.flux_dn_layer_top) {
        SSB_FL(f, flux_dn_layer_top, il) = vsum(dn_below, 0, n);
        SSB_FL(f, flux_up_layer_top, il) = vsum(up_below, 0, n);
        SSB_FL(f, flux_dn_layer_base, il) = vsum(dn_above, 0, n);
        SSB_FL(f, flux_up_layer_base, il) = vsum(up_above, 0, n);
      }
      L.load(oIF, n * n, jl, R);
      for (int i = 0; i < n; ++i) tmpv[i] = dn_below[i] + up_above[i];
      mat_vec(n, n, R, tmpv, iflux);
      if (internal) {
        L.load(oIsrc, n, jl, tmpv);
        for (int i = 0; i < n; ++i) iflux[i] = iflux[i] + tmpv[i];
        L.load(oBook, 3 * d + 1, jl, book);
      }
      auto sum_over_mu = [&](int r) {
        double s = 0.0;
        for (int js = 0; js < ns; ++js) s += iflux[r * ns + js] * (1.0 / a.lg.mu[js]);
        return s;
      };
      auto sum_tan = [&](int r) {
        double s = 0.0;
        for (int js = 0; js < ns; ++js) s += iflux[r * ns + js] * a.lg.tan_ang[js];
        return s;
      };
      const double dz = a.cp.dz[il];
      const double air_abs = SSB_LAY(a.lw.air_ext, g, il) * (1.0 - SSB_LAY(a.lw.air_ssa, g, il));
      if (internal)
        SSB_FL(f, clear_air_abs, il) = SSB_FL(f, clear_air_abs, il) + air_abs * sum_over_mu(0) - book[0] * dz;
      else
        SSB_FL(f, clear_air_abs, il) = SSB_FL(f, clear_air_abs, il) + air_abs * sum_over_mu(0);
      if (nreg > 1) {
        const double vabs = ve * (1.0 - SSB_LAY(a.lw.veg_ssa, g, il));
        for (int r = 1; r < nreg; ++r) {
          if (internal) {
            SSB_FL(f, veg_air_abs, il) = SSB_FL(f, veg_air_abs, il) + air_abs * sum_over_mu(r) - book[d + r] * dz;
            SSB_FL(f, veg_abs, il) =
                SSB_FL(f, veg_abs, il) + vabs * sum_over_mu(r) * gm.od_scaling[r] - book[2 * d + r] * dz;
          } else {
            SSB_FL(f, veg_air_abs, il) = SSB_FL(f, veg_air_abs, il) + air_abs * sum_over_mu(r);
            SSB_FL(f, veg_abs, il) = SSB_FL(f, veg_abs, il) + vabs * sum_over_mu(r) * gm.od_scaling[r];
          }
        }
      }
      if (c.urban) {
        for (int r = 0; r < nreg; ++r) SSB_FL(f, wall_in, il) = SSB_FL(f, wall_in, il) + gm.f_wall[r] * sum_tan(r);
        const double wemis = SSB_LAY(a.lw.wall_emissivity, g, il);
        if (internal)
          SSB_FL(f, wall_net, il) = SSB_FL(f, wall_in, il) * wemis - book[3 * d] * dz;
        else
          SSB_FL(f, wall_net, il) = SSB_FL(f, wall_in, il) * wemis;
      }
    }
    SSB_FC(f, ground_dn) = vsum(dn_above, 0, n);
    SSB_FC(f, ground_net) = SSB_FC(f, ground_dn) - vsum(up_above, 0, n);
    // forest_lw:687-694 accumulates the normalised pass into lw_internal as well
    const ssb200_canopy_flux &tgt = (internal || c.urban) ? f : fint;
    for (int r = 0; r < nreg; ++r)
      for (int js = 0; js < ns; ++js) {
        const int i = js + r * ns;
        SSB_FC(tgt, ground_vertical_diff) =
            SSB_FC(tgt, ground_vertical_diff) + (dn_above[i] + up_above[i]) * a.lg.tan_ang[js] / SSB_PI;
      }
  }
}

// ---------------------------------------------------------------------------
// Flat tiles and single-layer urban models: one thread per (column, interval)
// ---------------------------------------------------------------------------
struct SurfaceArgs {
  int ncols, nsw, nlw, do_sw, do_lw, use_sw_direct_albedo;
  double min_veg, min_bld;
  const int *cols;  // columns of type Flat / SimpleUrban / InfiniteStreet
  const int *nlay, *istartlay, *irep;
  ssb200_canopy_properties cp;
  ssb200_sw_spectral_properties sw;
  ssb200_lw_spectral_properties lw;
  ssb200_boundary_conds_out bc;
  ssb200_canopy_flux sw_dir, sw_diff, lw_int, lw_norm;
};

SSB_HD inline void surface_column_sw(const SurfaceArgs &a, int ic, int g) {
  const int col = a.cols[ic], nspec = a.nsw;
  const int irep = a.irep[col];
  const ssb200_canopy_flux &fd = a.sw_dir, &ff = a.sw_diff;
  const double galb = a.sw.ground_albedo[(size_t)g + (size_t)nspec * col];
  const double galb_dir = (a.use_sw_direct_albedo ? a.sw.ground_albedo_dir : a.sw.ground_albedo)[(size_t)g + (size_t)nspec * col];
  if (irep == SSB200_TILE_FLAT) {  // radsurf_interface.F90:130-154
    a.bc.sw_albedo[(size_t)g + (size_t)nspec * col] = galb;
    a.bc.sw_albedo_dir[(size_t)g + (size_t)nspec * col] = galb_dir;
    SSB_FC(fd, ground_dn_dir) = 1.0;
    SSB_FC(fd, ground_dn) = 1.0;
    SSB_FC(fd, ground_net) = 1.0 - galb_dir;
    SSB_FC(fd, ground_vertical_diff) = 0.5 * galb_dir;
    SSB_FC(fd, top_dn_dir) = 1.0;
    SSB_FC(fd, top_dn) = 1.0;
    SSB_FC(fd, top_net) = 1.0 - galb_dir;
    SSB_FC(ff, ground_dn_dir) = 0.0;
    SSB_FC(ff, ground_dn) = 1.0;
    SSB_FC(ff, ground_net) = 1.0 - galb;
    SSB_FC(ff, ground_vertical_diff) = 0.5 * (1.0 + galb);
    SSB_FC(ff, top_dn_dir) = 0.0;
    SSB_FC(ff, top_dn) = 1.0;
    SSB_FC(ff, top_net) = 1.0 - galb;
    return;
  }
  // simple_urban_sw (radsurf_simple_urban_sw.F90:28-294).  The reference indexes some
  // (nspec,ncol) members with the LAYER index (:193,219,253-256), which is only defined when
  // istartlay(j) = j (every earlier column has exactly one layer, as in test/single_layer): the
  // column index is used here - equal whenever the reference is well defined, in bounds otherwise.
  const int il = a.istartlay[col] - 1;
  const int nlay = a.nlay[col];
  const double cos_sza = a.cp.cos_sza[col];
  zero_column(fd, nspec, g, col, il, nlay, g == 0);
  zero_column(ff, nspec, g, col, il, nlay, g == 0);
  if (!(cos_sza > 0.0)) return;
  const bool inf = (irep == SSB200_TILE_INFINITE_STREET);
  const double dz = a.cp.dz[il], bf = a.cp.building_fraction[il], bs = a.cp.building_scale[il];
  const double npw = (bf > a.min_bld) ? 4.0 * bf / bs : 0.0;
  double vgs, vww, vdg;
  if (inf)
    view_factors(true, dz / (2.0 * (1.0 - bf) / npw), true, cos_sza, vgs, vww, vdg);
  else
    view_factors(false, dz / (SSB_PI * (1.0 - bf) / npw), true, cos_sza, vgs, vww, vdg);
  const double vdw = 1.0 - vdg, vwg = 0.5 * (1.0 - vww), vgw = 1.0 - vgs;
  const double ralb = SSB_LAY(a.sw.roof_albedo, g, il), walb = SSB_LAY(a.sw.wall_albedo, g, il);
  double im[4] = {1.0, -vgw * galb, -vwg * walb, 1.0 - vww * walb};  // column-major
  double srcv[2], sol[2], wk[4];
  srcv[0] = 0.0;
  srcv[1] = (vdw + galb_dir * vdg * vgw) * (1.0 - bf);
  solve_vec(2, im, srcv, sol, wk);
#define XC(f, member, c_) (f.member[(size_t)g + (size_t)nspec * (c_)])
  XC(fd, ground_dn_dir, col) = vdg * (1.0 - bf);
  XC(fd, ground_dn, col) = XC(fd, ground_dn_dir, col) + sol[0];
  XC(fd, ground_net, col) = XC(fd, ground_dn_dir, col) * (1.0 - galb_dir) + sol[0] * (1.0 - galb);
  if (g == 0) fd.ground_sunlit_frac[col] = vdg;
  XC(fd, roof_in_dir, il) = bf;
  XC(fd, roof_in, il) = bf;
  XC(fd, roof_net, il) = bf * (1.0 - ralb);
  XC(fd, wall_in_dir, il) = vdw * (1.0 - bf);
  XC(fd, wall_in, il) = sol[1];
  XC(fd, wall_net, il) = XC(fd, wall_in, il) * (1.0 - walb);
  if (g == 0) {
    fd.roof_sunlit_frac[il] = 1.0;
    const double tan_sza = sqrt(1.0 / (cos_sza * cos_sza) - 1.0);
    fd.wall_sunlit_frac[il] = 0.5 * vdw / (dmax(tan_sza, 1.0e-6) * npw * dz / (SSB_PI * (1.0 - bf)));
  }
  XC(fd, top_dn_dir, col) = 1.0;
  XC(fd, top_dn, col) = 1.0;
  XC(fd, top_net, col) = 1.0 - bf * ralb - (XC(fd, ground_dn, col) - XC(fd, ground_net, col)) * vgs -
                         (XC(fd, wall_in, il) - XC(fd, wall_net, il)) * vwg;
  if (fd.flux_dn_layer_top) {
    XC(fd, flux_dn_dir_layer_top, il) = (1.0 - bf);
    XC(fd, flux_dn_layer_top, il) = (1.0 - bf);
    XC(fd, flux_up_layer_top, il) = (XC(fd, ground_dn, col) - XC(fd, ground_net, col)) * vgs +
                                    (XC(fd, wall_in, il) - XC(fd, wall_net, il)) * vwg;
    XC(fd, flux_dn_dir_layer_base, il) = XC(fd, ground_dn_dir, col);
    XC(fd, flux_dn_layer_base, il) = XC(fd, ground_dn, col);
    XC(fd, flux_up_layer_base, il) = XC(fd, ground_dn, col) - XC(fd, ground_net, col);
  }
  srcv[0] = vgs * (1.0 - bf);
  srcv[1] = vgw * (1.0 - bf);
  solve_vec(2, im, srcv, sol, wk);
  XC(ff, ground_dn_dir, col) = 0.0;
  XC(ff, ground_dn, col) = sol[0];
  XC(ff, ground_net, col) = XC(ff, ground_dn, col) * (1.0 - galb);
  XC(ff, roof_in, il) = bf;
  XC(ff, roof_net, il) = bf * (1.0 - ralb);
  XC(ff, wall_in, il) = sol[1];
  XC(ff, wall_net, il) = XC(ff, wall_in, il) * (1.0 - walb);
  XC(ff, top_dn_dir, col) = 0.0;
  XC(ff, top_dn, col) = 1.0;
  XC(ff, top_net, col) = 1.0 - bf * ralb - (XC(ff, ground_dn, col) - XC(ff, ground_net, col)) * vgs -
                         (XC(ff, wall_in, il) - XC(ff, wall_net, il)) * vwg;
  if (ff.flux_dn_layer_top) {
    XC(ff, flux_dn_layer_top, il) = (1.0 - bf);
    XC(ff, flux_up_layer_top, il) = (XC(ff, ground_dn, col) - XC(ff, ground_net, col)) * vgs +
                                    (XC(ff, wall_in, il) - XC(ff, wall_net, il)) * vwg;
    XC(ff, flux_dn_layer_base, il) = XC(ff, ground_dn, col);
    XC(ff, flux_up_layer_base, il) = XC(ff, ground_dn, col) - XC(ff, ground_net, col);
  }
}

SSB_HD inline void surface_column_lw(const SurfaceArgs &a, int ic, int g) {
  const int col = a.cols[ic], nspec = a.nlw;
  const int irep = a.irep[col];
  const ssb200_canopy_flux &fi = a.lw_int, &fn = a.lw_norm;
  const double gemis = a.lw.ground_emissivity[(size_t)g + (size_t)nspec * col];
  const double gemission = a.lw.ground_emission[(size_t)g + (size_t)nspec * col];
  if (irep == SSB200_TILE_FLAT) {  // radsurf_interface.F90:156-172
    a.bc.lw_emissivity[(size_t)g + (size_t)nspec * col] = gemis;
    a.bc.lw_emission[(size_t)g + (size_t)nspec * col] = gemission;
    SSB_FC(fi, ground_dn) = 0.0;
    SSB_FC(fi, ground_net) = -gemission;
    SSB_FC(fi, ground_vertical_diff) = 0.5 * gemission;
    SSB_FC(fi, top_dn) = 0.0;
    SSB_FC(fi, top_net) = -gemission;
    SSB_FC(fn, ground_dn) = 1.0;
    SSB_FC(fn, ground_net) = gemis;
    SSB_FC(fn, ground_vertical_diff) = 0.5 * (2.0 - gemis);
    SSB_FC(fn, top_dn) = 1.0;
    SSB_FC(fn, top_net) = gemis;
    return;
  }
  // simple_urban_lw (radsurf_simple_urban_lw.F90:28-257)
  const int il = a.istartlay[col] - 1;
  const int nlay = a.nlay[col];
  zero_column(fn, nspec, g, col, il, nlay, g == 0);
  zero_column(fi, nspec, g, col, il, nlay, g == 0);
  const bool inf = (irep == SSB200_TILE_INFINITE_STREET);
  const double dz = a.cp.dz[il], bf = a.cp.building_fraction[il], bs = a.cp.building_scale[il];
  const double npw = (bf > a.min_bld) ? 4.0 * bf / bs : 0.0;
  double vgs, vww, vdg;
  if (inf)
    view_factors(true, dz / (2.0 * (1.0 - bf) / npw), false, 1.0, vgs, vww, vdg);
  else
    view_factors(false, dz / (SSB_PI * (1.0 - bf) / npw), false, 1.0, vgs, vww, vdg);
  const double vwg = 0.5 * (1.0 - vww), vgw = 1.0 - vgs;
  const double remis = SSB_LAY(a.lw.roof_emissivity, g, il), remission = SSB_LAY(a.lw.roof_emission, g, il);
  const double wemis = SSB_LAY(a.lw.wall_emissivity, g, il), wemission = SSB_LAY(a.lw.wall_emission, g, il);
  // interaction_matrix(2,2) uses the ground emissivity in the reference (simple_urban_lw:157)
  double im[4] = {1.0, -vgw * (1.0 - gemis), -vwg * (1.0 - wemis), 1.0 - vww * (1.0 - gemis)};
  double srcv[2], sol[2], wk[4];
  srcv[0] = vwg * wemission * npw * dz;
  srcv[1] = vgw * gemission * (1.0 - bf) + vww * wemission * npw * dz;
  solve_vec(2, im, srcv, sol, wk);
  XC(fi, ground_dn, col) = sol[0];
  XC(fi, ground_net, col) = sol[0] * gemis - gemission * (1.0 - bf);
  XC(fi, roof_in, il) = 0.0;
  XC(fi, roof_net, il) = -bf * remission;
  XC(fi, wall_in, il) = sol[1];
  XC(fi, wall_net, il) = sol[1] * wemis - wemission * npw * dz;
  XC(fi, top_dn, col) = 0.0;
  XC(fi, top_net, col) = -bf * remission - (XC(fi, ground_dn, col) - XC(fi, ground_net, col)) * vgs -
                         (XC(fi, wall_in, il) - XC(fi, wall_net, il)) * vwg;
  if (fi.flux_dn_layer_top) {
    XC(fi, flux_dn_layer_top, il) = 0.0;
    XC(fi, flux_up_layer_top, il) = (XC(fi, ground_dn, col) - XC(fi, ground_net, col)) * vgs +
                                    (XC(fi, wall_in, il) - XC(fi, wall_net, il)) * vwg;
    XC(fi, flux_dn_layer_base, il) = XC(fi, ground_dn, col);
    XC(fi, flux_up_layer_base, il) = XC(fi, ground_dn, col) - XC(fi, ground_net, col);
  }
  srcv[0] = vgs * (1.0 - bf);
  srcv[1] = vgw * (1.0 - bf);
  solve_vec(2, im, srcv, sol, wk);
  XC(fn, ground_dn, col) = sol[0];
  XC(fn, ground_net, col) = XC(fn, ground_dn, col) * gemis;
  XC(fn, roof_in, il) = bf;
  XC(fn, roof_net, il) = bf * remis;
  XC(fn, wall_in, il) = sol[1];
  XC(fn, wall_net, il) = XC(fn, wall_in, il) * wemis;
  XC(fn, top_dn, col) = 1.0;
  XC(fn, top_net, col) = 1.0 - bf * (1.0 - remis) - (XC(fn, ground_dn, col) - XC(fn, ground_net, col)) * vgs -
                         (XC(fn, wall_in, il) - XC(fn, wall_net, il)) * vwg;
  if (fn.flux_dn_layer_top) {
    XC(fn, flux_dn_layer_top, il) = 1.0 - bf;
    XC(fn, flux_up_layer_top, il) = (XC(fn, ground_dn, col) - XC(fn, ground_net, col)) * vgs +
                                    (XC(fn, wall_in, il) - XC(fn, wall_net, il)) * vwg;
    XC(fn, flux_dn_layer_base, il) = XC(fn, ground_dn, col);
    XC(fn, flux_up_layer_base, il) = XC(fn, ground_dn, col) - XC(fn, ground_net, col);
  }
#undef XC
}

}  // namespace ssb
