// ssb_fast_sweeps.cuh - register-resident adding sweeps: one thread per
// (column, interval) with compile-time (NREG regions, NS streams, URBAN).
//
// Same recurrences and outputs as column_sweeps_sw/_lw of ssb_solver.cuh
// (radsurf_urban_sw.F90:591-984, radsurf_urban_lw.F90:552-858 and the forest
// equivalents), organised around HBM traffic, which bounds these kernels:
//  * only a_above and d_above (or source_above) are kept per interface (the
//    LU factors of the denominator I - a_above R are rebuilt in the downward
//    pass from a_above and R, which it loads anyway); the "below" albedo
//    matrices (which carry the extra roof region) are never formed in the
//    downward pass - their action on a flux vector is evaluated as
//      a_below x = R x + T D^-1 (a_above (T x))   (+ the roof block),
//    and likewise for d_below and source_below (SURVEY F6);
//  * the overlap matrices U, V are recomputed from the region fractions of the
//    two adjacent layers instead of being stored;
//  * the two downward passes of the reference (direct and diffuse source in
//    the shortwave, internal emission and incoming in the longwave) run
//    together, so every layer matrix is streamed from HBM once per layer and
//    each loaded element feeds both passes;
//  * the state carried up the column (a_above, d_above) lives in a per-thread
//    slice of shared memory (`StateMem`), which keeps the upward sweep inside
//    the register file.
#pragma once
#include "ssb_fast_layer.cuh"
#include "ssb_sweep_blocks.cuh"

namespace ssb {

// One scratch area (layer or interface) as seen by the calling problem: `base` points at
// element 0 of level 0, levels are `lev_stride` doubles apart and element e sits at the
// compile-time offset e * kScratchTile, so a layer is addressed from one register pair.
struct Scr {
  double *base;
  size_t lev_stride;
  SSB_HDI Scr(double *area, int nlev, int nelem, int q)
      : base(area + sidx(0, 0, nlev, nelem, q)), lev_stride((size_t)nelem * kScratchTile) {}
  // The scratch is streamed (every element is used once or twice, hundreds of megabytes apart):
  // evict-first loads and stores keep it from flushing the partially written sectors of the
  // per-column output arrays out of L2.
  SSB_HDI double ld(int e, int lev) const {
#if defined(__CUDA_ARCH__)
    return __ldcs(base + (size_t)lev * lev_stride + (size_t)e * kScratchTile);
#else
    return base[(size_t)lev * lev_stride + (size_t)e * kScratchTile];
#endif
  }
  SSB_HDI double ldp(int e, int lev, bool keep) const {  // structural zeros are not loaded
    double v = 0.0;
    if (keep) v = ld(e, lev);
    return v;
  }
  SSB_HDI void prefetch(int e, int lev) const {  // into L2 (no register, no scoreboard entry)
#if defined(__CUDA_ARCH__)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(base + (size_t)lev * lev_stride + (size_t)e * kScratchTile));
#else
    (void)e;
    (void)lev;
#endif
  }
  SSB_HDI void st(int e, int lev, double v) const {
#if defined(__CUDA_ARCH__)
    __stcs(base + (size_t)lev * lev_stride + (size_t)e * kScratchTile, v);
#else
    base[(size_t)lev * lev_stride + (size_t)e * kScratchTile] = v;
#endif
  }
};

// A layer that solves only a sub-block of its regions ("segment" 1: clear region, 2: vegetated
// regions; radsurf_urban_sw.F90:512-583) leaves the rest of its matrices zero.  The layer
// kernels do not write those zeros and the sweeps do not load them: an element is loaded when
// the segment keeps its class (0: couples the clear region with a vegetated one, 1: inside the
// clear block, 2: inside the vegetated block).  KIND: 0 = streams x streams (n x n),
// 1 = streams x regions (n x d), 2 = regions x regions (d x d), 3 = vector over streams.
struct SegKeep {
  bool k[3];
};
SSB_HDI SegKeep seg_keep(int seg) { return SegKeep{{seg == 0, seg != 2, seg != 1}}; }
template <int KIND, int NS>
SSB_HD constexpr int seg_class(int i, int j) {
  return KIND == 3 ? (i / NS == 0 ? 1 : 2)
                   : ((KIND == 2 ? i : i / NS) == 0 && (KIND == 0 ? j / NS : j) == 0)
                         ? 1
                         : ((KIND == 2 ? i : i / NS) > 0 && (KIND == 0 ? j / NS : j) > 0) ? 2 : 0;
}

// L2 prefetch of the NA x NA block at offset `off` (n x n layout) of level `lev`
template <int n, int NA, int I0>
SSB_HDI void prefetch_block(const Scr &S, int off, int lev) {
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) S.prefetch(off + (I0 + i) + n * (I0 + j), lev);
  }
}
#ifndef SSB_SWEEP_PREFETCH
#define SSB_SWEEP_PREFETCH 0
#endif

// (V (x) I_NS) x : below-interface vector (NRB*NS) from the above-interface one (NREG*NS)
template <int NREG, int NRB, int NS>
SSB_HDI void expand_down(const double *V, const double *x, double *y) {
  SSB_UNROLL
  for (int lo = 0; lo < NRB; ++lo) {
    SSB_UNROLL
    for (int js = 0; js < NS; ++js) {
      double s = 0.0;
      SSB_UNROLL
      for (int up = 0; up < NREG; ++up) s = fma(V[lo + NRB * up], x[up * NS + js], s);
      y[lo * NS + js] = s;
    }
  }
}

// y1 += A x1, y2 += A x2 with A (R x C) streamed once from scratch
template <int R, int C, int KIND = -1, int NS = 1>
SSB_HDI void smv2(const Scr &S, int e0, int lev, const double *x1, const double *x2, double *y1, double *y2,
                  const SegKeep &sk = SegKeep{{true, true, true}}) {
  SSB_UNROLL
  for (int j = 0; j < C; ++j) {
    SSB_UNROLL
    for (int i = 0; i < R; ++i) {
      const double a = (KIND < 0) ? S.ld(e0 + i + R * j, lev)
                                  : S.ldp(e0 + i + R * j, lev, sk.k[seg_class<(KIND < 0 ? 0 : KIND), NS>(i, j)]);
      y1[i] = fma(a, x1[j], y1[i]);
      y2[i] = fma(a, x2[j], y2[i]);
    }
  }
}
template <int R, int C, int KIND = -1, int NS = 1>
SSB_HDI void smv1(const Scr &S, int e0, int lev, const double *x, double *y,
                  const SegKeep &sk = SegKeep{{true, true, true}}) {
  SSB_UNROLL
  for (int j = 0; j < C; ++j) {
    SSB_UNROLL
    for (int i = 0; i < R; ++i) {
      const double a = (KIND < 0) ? S.ld(e0 + i + R * j, lev)
                                  : S.ldp(e0 + i + R * j, lev, sk.k[seg_class<(KIND < 0 ? 0 : KIND), NS>(i, j)]);
      y[i] = fma(a, x[j], y[i]);
    }
  }
}

// overlap matrices of the interface above layer jl of the column starting at packed layer il1
// (radsurf_overlap.F90), from the region fractions of the two adjacent layers
template <int NREG, bool URBAN, bool LW>
SSB_HDI void overlap_above(const ClassArgs &a, int il1, int nlay, int jl, double *U, double *V) {
  const bool veg = NREG > 1 || !URBAN;
  const int ls = layer_step(a);
  double fb[3] = {0.0, 0.0, 0.0}, fa[3] = {0.0, 0.0, 0.0};
  {
    const int il = il1 + jl * ls;
    region_fractions_t<NREG, URBAN, LW>(URBAN ? a.cp.building_fraction[il] : 0.0,
                                        (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il] : 0.0, fb);
  }
  const bool top = jl + 1 >= nlay;
  if (!top) {
    const int il = il1 + (jl + 1) * ls;
    region_fractions_t<NREG, URBAN, LW>(URBAN ? a.cp.building_fraction[il] : 0.0,
                                        (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il] : 0.0, fa);
  }
  overlap_fast<NREG, URBAN>(fb, fa, top, a.cfg.min_veg, U, V);
}

// a_above(next)[(u,jt),(up,js)] = sum_{lo,lo'} U[u,lo] V[lo',up] Ab[(lo,jt),(lo',js)] + roof term,
// evaluated per stream pair as a 3x3 "region sandwich" and written to the state slice
template <int NREG, int NRB, int NS>
SSB_HDI void overlap_matrix(const double *Ab, const double *rb, const double *U, const double *V,
                            const StateMem &st, int o) {
  constexpr int n = NREG * NS;
  SSB_UNROLL
  for (int jt = 0; jt < NS; ++jt) {
    SSB_UNROLL
    for (int js = 0; js < NS; ++js) {
      double BV[NREG * NREG];  // [lo + NREG*up]
      SSB_UNROLL
      for (int up = 0; up < NREG; ++up) {
        SSB_UNROLL
        for (int lo = 0; lo < NREG; ++lo) {
          double s = 0.0;
          SSB_UNROLL
          for (int l2 = 0; l2 < NREG; ++l2) s = fma(Ab[(lo * NS + jt) + n * (l2 * NS + js)], V[l2 + NRB * up], s);
          BV[lo + NREG * up] = s;
        }
      }
      SSB_UNROLL
      for (int up = 0; up < NREG; ++up) {
        SSB_UNROLL
        for (int u = 0; u < NREG; ++u) {
          double s = 0.0;
          SSB_UNROLL
          for (int lo = 0; lo < NREG; ++lo) s = fma(U[u + NREG * lo], BV[lo + NREG * up], s);
          if (NRB > NREG) s = fma(U[u + NREG * NREG] * rb[jt], V[NREG + NRB * up], s);
          st(o + (u * NS + jt) + n * (up * NS + js)) = s;
        }
      }
    }
  }
}

// canopy_flux%zero semantics without writing twice: the sweeps assign every member they
// own, so only the members of OTHER tile types (and the direct-only members of the
// diffuse object) are cleared here (radsurf_canopy_flux.F90:286-341).
template <int NREG, bool URBAN>
SSB_HDI void zero_unwritten_sw(const ssb200_canopy_flux &f, int nspec, int g, int col, int il1, int nlay, bool own,
                               bool direct, int ls = 1) {
  auto zl = [&](double *p) {
    if (p)
      for (int l = 0; l < nlay; ++l) p[(size_t)g + (size_t)nspec * (il1 + l * ls)] = 0.0;
  };
  auto zs = [&](double *p) {
    if (p && own)
      for (int l = 0; l < nlay; ++l) p[il1 + l * ls] = 0.0;
  };
  if (!URBAN) {
    zl(f.roof_in);
    zl(f.roof_net);
    zl(f.wall_in);
    zl(f.wall_net);
    zl(f.roof_in_dir);
    zl(f.wall_in_dir);
    zs(f.roof_sunlit_frac);
    zs(f.wall_sunlit_frac);
  }
  if (NREG == 1) {
    zl(f.veg_abs);
    zl(f.veg_air_abs);
    zl(f.veg_abs_dir);
    zs(f.veg_sunlit_frac);
  }
  if (!direct) {
    zl(f.roof_in_dir);
    zl(f.wall_in_dir);
    zl(f.veg_abs_dir);
    zl(f.flux_dn_dir_layer_top);
    zl(f.flux_dn_dir_layer_base);
    zs(f.roof_sunlit_frac);
    zs(f.wall_sunlit_frac);
    zs(f.veg_sunlit_frac);
    if (own && f.ground_sunlit_frac) f.ground_sunlit_frac[col] = 0.0;
  }
}
template <int NREG, bool URBAN>
SSB_HDI void zero_unwritten_lw(const ssb200_canopy_flux &f, int nspec, int g, int col, int il1, int nlay, int ls = 1) {
  auto zl = [&](double *p) {
    if (p)
      for (int l = 0; l < nlay; ++l) p[(size_t)g + (size_t)nspec * (il1 + l * ls)] = 0.0;
  };
  if (!URBAN) {
    zl(f.roof_in);
    zl(f.roof_net);
    zl(f.wall_in);
    zl(f.wall_net);
  }
  if (NREG == 1) {
    zl(f.veg_abs);
    zl(f.veg_air_abs);
  }
  // direct-only members exist only if the caller allocated a LW object with use_direct
  zl(f.roof_in_dir);
  zl(f.wall_in_dir);
  zl(f.veg_abs_dir);
  zl(f.flux_dn_dir_layer_top);
  zl(f.flux_dn_dir_layer_base);
  if (f.ground_dn_dir) f.ground_dn_dir[(size_t)g + (size_t)nspec * col] = 0.0;
  if (f.top_dn_dir) f.top_dn_dir[(size_t)g + (size_t)nspec * col] = 0.0;
  if (g == 0) {
    if (f.ground_sunlit_frac) f.ground_sunlit_frac[col] = 0.0;
    for (int l = 0; l < nlay; ++l) {
      if (f.roof_sunlit_frac) f.roof_sunlit_frac[il1 + l * ls] = 0.0;
      if (f.wall_sunlit_frac) f.wall_sunlit_frac[il1 + l * ls] = 0.0;
      if (f.veg_sunlit_frac) f.veg_sunlit_frac[il1 + l * ls] = 0.0;
    }
  }
}

// ===========================================================================
// Shortwave
// ===========================================================================
template <int NREG, int NS, bool URBAN>
struct SwSweepLayout {
  static constexpr int n = NREG * NS, d = NREG;
  static constexpr int oR = 0, oT = n * n, oIdiff = 2 * n * n, oSup = 3 * n * n, oSdn = oSup + n * d,
                       oIdd = oSdn + n * d, oE = oIdd + n * d, oIdir = oE + d * d;
  static constexpr int oGeo = oIdir + d * d;                      // geometry block (fast_prepare_level)
  static constexpr int oAa = 0, oDa = n * n;  // interface scratch of the fast path (state_doubles per level)
  static constexpr int NRB = URBAN ? NREG + 1 : NREG, m = NRB * NS;
  static constexpr int state_doubles = fast_sw_sweep_elems(n, d);
  // block of a layer that solves only its vegetated regions (segment 2)
  static constexpr int vegNA = NREG > 1 ? n - NS : n, vegI0 = NREG > 1 ? NS : 0;
};

template <int NREG, int NS, bool URBAN>
SSB_HD inline void fast_column_sweeps_sw(const ClassArgs &a, int q, const StateMem &st) {
  typedef SwSweepLayout<NREG, NS, URBAN> Lay;
  constexpr int n = NREG * NS, d = NREG, NRB = URBAN ? NREG + 1 : NREG, m = NRB * NS;
  const SolveCfg &c = a.cfg;
  const int nspec = c.nspec;
  const int ic = q / nspec, g = q % nspec;
  const int col = a.cols[ic];
  const int nlay = a.nlay[col], il1 = layer_index(a, ic, col, 0), ls = layer_step(a);
  const ssb200_canopy_flux &fdir = a.f1, &fdif = a.f2;
  const double cos_sza = a.cp.cos_sza[col];
  int itransp = 0;
  if (nspec > 1) {
    double best = 0.0;
    for (int gg = 0; gg < nspec; ++gg) {
      double od = 0.0;
      for (int l = 0; l < nlay; ++l) od += a.sw.air_ext[(size_t)gg + (size_t)nspec * (il1 + l * ls)] * a.cp.dz[il1 + l * ls];
      if (gg == 0 || od < best) {
        best = od;
        itransp = gg;
      }
    }
  }
  const bool own = (g == itransp);
  if (!(cos_sza > 0.0)) {  // night: every member of the column is zero (radsurf_interface.F90:193-196)
    zero_column(fdir, nspec, g, col, il1, nlay, own, ls);
    zero_column(fdif, nspec, g, col, il1, nlay, own, ls);
    return;
  }
  zero_unwritten_sw<NREG, URBAN>(fdir, nspec, g, col, il1, nlay, own, true, ls);
  zero_unwritten_sw<NREG, URBAN>(fdif, nspec, g, col, il1, nlay, own, false, ls);
  const double zcos = URBAN ? dmax(cos_sza, 1.0e-6) : cos_sza;
  const double sin0 = URBAN ? sqrt(1.0 - zcos * zcos) : 0.0;
  const double galb = a.sw.ground_albedo[(size_t)g + (size_t)nspec * col];
  const double galb_dir =
      (a.use_sw_direct_albedo ? a.sw.ground_albedo_dir : a.sw.ground_albedo)[(size_t)g + (size_t)nspec * col];
  double hw[NS], mu_inv[NS], tang[NS];
  SSB_UNROLL
  for (int js = 0; js < NS; ++js) {
    hw[js] = a.lg.hweight[js];
    mu_inv[js] = 1.0 / a.lg.mu[js];
    tang[js] = a.lg.tan_ang[js];
  }
  const Scr L(a.layer, a.lmax, a.ne_layer, q);
  const Scr W(a.sweep, a.lmax + 1, a.ne_sweep, q);
  // the upwelling flux outside the block a layer solves is only needed for the flux profiles (and at
  // the ground: level 0 is always stored and read in full)
  const bool full_ua = fdir.flux_dn_layer_top != nullptr || fdif.flux_dn_layer_top != nullptr;

  // ---- upward sweep: state = [a_above (n x n) | d_above (n x d)] ------------
  SSB_UNROLL
  for (int i = 0; i < Lay::state_doubles; ++i) st(i) = 0.0;
  SSB_UNROLL
  for (int r = 0; r < NREG; ++r) {
    SSB_UNROLL
    for (int jt = 0; jt < NS; ++jt) {
      st(Lay::oDa + (jt + r * NS) + n * r) = zcos * galb_dir * hw[jt];
      SSB_UNROLL
      for (int jf = 0; jf < NS; ++jf) st((jt + r * NS) + n * (jf + r * NS)) = galb * hw[jt];
    }
  }
  SSB_UNROLL
  for (int i = 0; i < Lay::state_doubles; ++i) W.st(i, 0, st(i));
  for (int jl = 0; jl < nlay; ++jl) {
    const int il = il1 + jl * ls;
    // the adding step on the block of regions the layer solves (ssb_sweep_blocks.cuh); with the columns
    // of the launch ordered by segment pattern the switch is uniform per warp
    const int seg = (int)L.ld(Lay::oGeo + 7, jl);
    if (SSB_SWEEP_PREFETCH && jl + 1 < nlay) {
      const int sn = (int)L.ld(Lay::oGeo + 7, jl + 1);
      if (NREG == 1 || sn == 0) {
        prefetch_block<n, n, 0>(L, Lay::oR, jl + 1);
        prefetch_block<n, n, 0>(L, Lay::oT, jl + 1);
      } else if (sn == 1) {
        prefetch_block<n, NS, 0>(L, Lay::oR, jl + 1);
        prefetch_block<n, NS, 0>(L, Lay::oT, jl + 1);
      }
    }
    double Ab[n * n], Db[n * d];
    if (NREG == 1 || seg == 0)
      sw_up_block<Lay, NREG, NS, n, 0>(st, L, jl, Ab, Db);
    else if (seg == 1)
      sw_up_block<Lay, NREG, NS, NS, 0>(st, L, jl, Ab, Db);
    else
      sw_up_block<Lay, NREG, NS, Lay::vegNA, Lay::vegI0>(st, L, jl, Ab, Db);
    double rb[NS], rd[NS];
    SSB_UNROLL
    for (int js = 0; js < NS; ++js) rb[js] = rd[js] = 0.0;
    if (URBAN) {
      const double ralb = SSB_LAY(a.sw.roof_albedo, g, il);
      const double ralb_dir = a.sw.roof_albedo_dir ? SSB_LAY(a.sw.roof_albedo_dir, g, il) : ralb;
      SSB_UNROLL
      for (int js = 0; js < NS; ++js) {
        rb[js] = ralb * hw[js];
        rd[js] = zcos * ralb_dir * hw[js];
      }
    }
    double U[12], V[12];
    overlap_above<NREG, URBAN, false>(a, il1, nlay, jl, U, V);
    overlap_matrix<NREG, NRB, NS>(Ab, rb, U, V, st, Lay::oAa);
    // d_above(next)[(u,jt), up] = sum U[u,lo] (Db V)[(lo,jt), up] + roof
    SSB_UNROLL
    for (int jt = 0; jt < NS; ++jt) {
      double DV[NREG * NREG];
      SSB_UNROLL
      for (int up = 0; up < NREG; ++up) {
        SSB_UNROLL
        for (int lo = 0; lo < NREG; ++lo) {
          double s = 0.0;
          SSB_UNROLL
          for (int l2 = 0; l2 < NREG; ++l2) s = fma(Db[(lo * NS + jt) + n * l2], V[l2 + NRB * up], s);
          DV[lo + NREG * up] = s;
        }
      }
      SSB_UNROLL
      for (int up = 0; up < NREG; ++up) {
        SSB_UNROLL
        for (int u = 0; u < NREG; ++u) {
          double s = 0.0;
          SSB_UNROLL
          for (int lo = 0; lo < NREG; ++lo) s = fma(U[u + NREG * lo], DV[lo + NREG * up], s);
          if (URBAN) s = fma(U[u + NREG * NREG] * rd[jt], V[NREG + NRB * up], s);
          st(Lay::oDa + (u * NS + jt) + n * up) = s;
        }
      }
    }
    // the state above the top layer is the top-of-canopy albedo (used from `st` below, never re-read);
    // a consumer layer that solves a sub-block gets only the entries it reads (interface_store_pruned)
    if (jl + 1 < nlay) {
      const int sn = (NREG == 1 || full_ua) ? 0 : (int)L.ld(Lay::oGeo + 7, jl + 1);
      if (sn == 0) {
        SSB_UNROLL
        for (int i = 0; i < Lay::state_doubles; ++i) W.st(i, jl + 1, st(i));
      } else if (sn == 1) {
        interface_store_pruned<Lay, n, NS, 0, 1, 0>(st, W, jl + 1);
      } else {
        interface_store_pruned<Lay, n, Lay::vegNA, Lay::vegI0, Lay::vegNA / NS, Lay::vegI0 / NS>(st, W, jl + 1);
      }
    }
  }
  double talb_diff = 0.0, talb_dir = 0.0;
  {
    SSB_UNROLL
    for (int i = 0; i < NS; ++i) {
      double s = 0.0;
      SSB_UNROLL
      for (int j = 0; j < NS; ++j) s = fma(st(i + n * j), hw[j], s);
      talb_diff += s;
    }
    double s = 0.0;
    SSB_UNROLL
    for (int js = 0; js < NS; ++js) s += st(Lay::oDa + js);
    talb_dir = s / zcos;
    a.bc.sw_albedo[(size_t)g + (size_t)nspec * col] = talb_diff;
    a.bc.sw_albedo_dir[(size_t)g + (size_t)nspec * col] = talb_dir;
  }

  // ---- downward sweep, direct (suffix d) and diffuse (suffix f) sources together ----
  double dir_above[d], xa_d[n], xa_f[n], ua_d[n], ua_f[n];
  SSB_UNROLL
  for (int i = 0; i < d; ++i) dir_above[i] = 0.0;
  SSB_UNROLL
  for (int i = 0; i < n; ++i) xa_d[i] = xa_f[i] = ua_d[i] = ua_f[i] = 0.0;
  dir_above[0] = 1.0 / zcos;
  SSB_UNROLL
  for (int js = 0; js < NS; ++js) xa_f[js] = hw[js];
  SSB_FC(fdir, top_dn_dir) = 1.0;
  SSB_FC(fdir, top_dn) = 1.0;
  SSB_FC(fdir, top_net) = 1.0 * (1.0 - talb_dir);
  SSB_FC(fdif, top_dn_dir) = 0.0;
  SSB_FC(fdif, top_dn) = 1.0;
  SSB_FC(fdif, top_net) = 1.0 - talb_diff;
  if (URBAN && own && fdir.roof_sunlit_frac && nlay > 0) fdir.roof_sunlit_frac[il1 + (nlay - 1) * ls] = 1.0;
  double flux_dn_dir_clear = 1.0 / zcos;
  for (int jl = nlay - 1; jl >= 0; --jl) {
    const int il = il1 + jl * ls;
    const int seg = (int)L.ld(Lay::oGeo + 7, jl);
    double f_wall[3], od_scaling[3];
    SSB_UNROLL
    for (int r = 0; r < 3; ++r) {
      f_wall[r] = L.ld(Lay::oGeo + r, jl);
      od_scaling[r] = L.ld(Lay::oGeo + 3 + r, jl);
    }
    const double f_wall_dir_clear = L.ld(Lay::oGeo + 6, jl);
    const bool veg = NREG > 1 || !URBAN;
    const double bf = URBAN ? a.cp.building_fraction[il] : 0.0;
    const double vf = (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il] : 0.0;
    const double ve = (veg && a.cp.veg_ext) ? a.cp.veg_ext[il] : 0.0;
    double xb_d[m], xb_f[m], dir_below[NRB];
    {
      double U[12], V[12];
      overlap_above<NREG, URBAN, false>(a, il1, nlay, jl, U, V);
      expand_down<NREG, NRB, NS>(V, xa_d, xb_d);
      expand_down<NREG, NRB, NS>(V, xa_f, xb_f);
      SSB_UNROLL
      for (int lo = 0; lo < NRB; ++lo) {
        double s = 0.0;
        SSB_UNROLL
        for (int up = 0; up < NREG; ++up) s = fma(V[lo + NRB * up], dir_above[up], s);
        dir_below[lo] = s;
      }
    }
    if (SSB_SWEEP_PREFETCH && jl > 0) {
      const int sn = (int)L.ld(Lay::oGeo + 7, jl - 1);
      prefetch_block<n, n, 0>(W, Lay::oAa, jl - 1);
      if (NREG == 1 || sn == 0) {
        prefetch_block<n, n, 0>(L, Lay::oT, jl - 1);
        prefetch_block<n, n, 0>(L, Lay::oR, jl - 1);
      } else if (sn == 1) {
        prefetch_block<n, NS, 0>(L, Lay::oT, jl - 1);
        prefetch_block<n, NS, 0>(L, Lay::oR, jl - 1);
      }
    }
    // the step on the block of regions the layer solves (ssb_sweep_blocks.cuh)
    double refl[n], ddir[d], ub_d[m], ub_f[m], if_d[n], if_f[n], idir[d];
    if (NREG == 1 || seg == 0)
      sw_down_block<Lay, NREG, NS, n, 0>(L, W, jl, xb_d, xb_f, dir_below, xa_d, xa_f, dir_above, ddir, refl, ub_d, ub_f,
                                         ua_d, ua_f, if_d, if_f, idir);
    else if (seg == 1) {
      if (full_ua || jl == 0)
        sw_down_block<Lay, NREG, NS, NS, 0, true>(L, W, jl, xb_d, xb_f, dir_below, xa_d, xa_f, dir_above, ddir, refl, ub_d,
                                                  ub_f, ua_d, ua_f, if_d, if_f, idir);
      else
        sw_down_block<Lay, NREG, NS, NS, 0, false>(L, W, jl, xb_d, xb_f, dir_below, xa_d, xa_f, dir_above, ddir, refl, ub_d,
                                                   ub_f, ua_d, ua_f, if_d, if_f, idir);
    } else {
      if (full_ua || jl == 0)
        sw_down_block<Lay, NREG, NS, Lay::vegNA, Lay::vegI0, true>(L, W, jl, xb_d, xb_f, dir_below, xa_d, xa_f, dir_above,
                                                                  ddir, refl, ub_d, ub_f, ua_d, ua_f, if_d, if_f, idir);
      else
        sw_down_block<Lay, NREG, NS, Lay::vegNA, Lay::vegI0, false>(L, W, jl, xb_d, xb_f, dir_below, xa_d, xa_f, dir_above,
                                                                   ddir, refl, ub_d, ub_f, ua_d, ua_f, if_d, if_f, idir);
    }
    SSB_UNROLL
    for (int i = n; i < m; ++i) ub_d[i] = ub_f[i] = 0.0;
    if (URBAN) {
      const double ralb = SSB_LAY(a.sw.roof_albedo, g, il);
      const double ralb_dir = a.sw.roof_albedo_dir ? SSB_LAY(a.sw.roof_albedo_dir, g, il) : ralb;
      double sroof_d = 0.0, sroof_f = 0.0, rup_d = 0.0, rup_f = 0.0;
      SSB_UNROLL
      for (int js = 0; js < NS; ++js) {
        sroof_d += xb_d[n + js];
        sroof_f += xb_f[n + js];
      }
      SSB_UNROLL
      for (int js = 0; js < NS; ++js) {
        ub_d[n + js] = ralb * hw[js] * sroof_d + zcos * ralb_dir * hw[js] * dir_below[NREG];
        ub_f[n + js] = ralb * hw[js] * sroof_f;
        rup_d += ub_d[n + js];
        rup_f += ub_f[n + js];
      }
      SSB_FL(fdir, roof_in_dir, il) = zcos * dir_below[NREG];
      SSB_FL(fdir, roof_in, il) = SSB_FL(fdir, roof_in_dir, il) + sroof_d;
      SSB_FL(fdir, roof_net, il) = SSB_FL(fdir, roof_in, il) - rup_d;
      SSB_FL(fdif, roof_in, il) = sroof_f;
      SSB_FL(fdif, roof_net, il) = sroof_f - rup_f;
    }
    if (fdir.flux_dn_layer_top || fdif.flux_dn_layer_top) {
      double s[8] = {0, 0, 0, 0, 0, 0, 0, 0}, sdb = 0.0, sda = 0.0;
      SSB_UNROLL
      for (int i = 0; i < n; ++i) {
        s[0] += xb_d[i];
        s[1] += xa_d[i];
        s[2] += ub_d[i];
        s[3] += ua_d[i];
        s[4] += xb_f[i];
        s[5] += xa_f[i];
        s[6] += ub_f[i];
        s[7] += ua_f[i];
      }
      SSB_UNROLL
      for (int i = 0; i < d; ++i) {
        sdb += dir_below[i];
        sda += dir_above[i];
      }
      if (fdir.flux_dn_layer_top) {
        SSB_FL(fdir, flux_dn_dir_layer_top, il) = zcos * sdb;
        SSB_FL(fdir, flux_dn_layer_top, il) = zcos * sdb + s[0];
        SSB_FL(fdir, flux_dn_dir_layer_base, il) = zcos * sda;
        SSB_FL(fdir, flux_dn_layer_base, il) = zcos * sda + s[1];
        SSB_FL(fdir, flux_up_layer_top, il) = s[2];
        SSB_FL(fdir, flux_up_layer_base, il) = s[3];
      }
      if (fdif.flux_dn_layer_top) {
        SSB_FL(fdif, flux_dn_layer_top, il) = s[4];
        SSB_FL(fdif, flux_dn_layer_base, il) = s[5];
        SSB_FL(fdif, flux_up_layer_top, il) = s[6];
        SSB_FL(fdif, flux_up_layer_base, il) = s[7];
      }
    }
    double smu_d[NREG], smu_f[NREG], stan_d[NREG], stan_f[NREG];
    SSB_UNROLL
    for (int r = 0; r < NREG; ++r) {
      smu_d[r] = smu_f[r] = stan_d[r] = stan_f[r] = 0.0;
      SSB_UNROLL
      for (int js = 0; js < NS; ++js) {
        smu_d[r] = fma(if_d[r * NS + js], mu_inv[js], smu_d[r]);
        smu_f[r] = fma(if_f[r * NS + js], mu_inv[js], smu_f[r]);
        stan_d[r] = fma(if_d[r * NS + js], tang[js], stan_d[r]);
        stan_f[r] = fma(if_f[r * NS + js], tang[js], stan_f[r]);
      }
    }
    const double air_ext = SSB_LAY(a.sw.air_ext, g, il);
    const double air_abs = air_ext * (1.0 - SSB_LAY(a.sw.air_ssa, g, il));
    SSB_FL(fdir, clear_air_abs, il) = air_abs * (idir[0] + smu_d[0]);
    SSB_FL(fdif, clear_air_abs, il) = air_abs * smu_f[0];
    if (NREG > 1) {
      const double vabs = ve * (1.0 - SSB_LAY(a.sw.veg_ssa, g, il));
      double air_d = 0.0, veg_d = 0.0, vdir = 0.0, air_f = 0.0, veg_f = 0.0;
      SSB_UNROLL
      for (int r = 1; r < NREG; ++r) {
        air_d += air_abs * (idir[r] + smu_d[r]);
        vdir += vabs * idir[r] * od_scaling[r];
        veg_d += vabs * (idir[r] + smu_d[r]) * od_scaling[r];
        air_f += air_abs * smu_f[r];
        veg_f += vabs * smu_f[r] * od_scaling[r];
      }
      SSB_FL(fdir, veg_air_abs, il) = air_d;
      SSB_FL(fdir, veg_abs, il) = veg_d;
      SSB_FL(fdir, veg_abs_dir, il) = vdir;
      SSB_FL(fdif, veg_air_abs, il) = air_f;
      SSB_FL(fdif, veg_abs, il) = veg_f;
    }
    if (URBAN) {
      const double walb = SSB_LAY(a.sw.wall_albedo, g, il);
      double win_dir = 0.0, win_d = 0.0, win_f = 0.0;
      SSB_UNROLL
      for (int r = 0; r < NREG; ++r) {
        win_dir += f_wall[r] * sin0 * idir[r];
        win_d += f_wall[r] * stan_d[r];
        win_f += f_wall[r] * stan_f[r];
      }
      SSB_FL(fdir, wall_in_dir, il) = win_dir;
      SSB_FL(fdir, wall_in, il) = win_dir + win_d;
      SSB_FL(fdir, wall_net, il) = (win_dir + win_d) * (1.0 - walb);
      SSB_FL(fdif, wall_in, il) = win_f;
      SSB_FL(fdif, wall_net, il) = win_f * (1.0 - walb);
    }
    {
      // spectrally independent sunlit fractions from the most transparent interval (urban_sw:805-848)
      const double nonb_here = URBAN ? 1.0 - bf : 1.0;
      double nonb_above = 1.0;
      if (URBAN && jl + 1 < nlay) nonb_above = 1.0 - a.cp.building_fraction[il + ls];
      if (URBAN) {
        const double roof_fraction = (jl == nlay - 1) ? bf : dmax(0.0, bf - a.cp.building_fraction[il + ls]);
        if (own && fdir.roof_sunlit_frac)
          fdir.roof_sunlit_frac[il] = SSB_FL(fdir, roof_in_dir, il) * nonb_above /
                                      (zcos * flux_dn_dir_clear * dmax(c.min_bld, roof_fraction));
        flux_dn_dir_clear = flux_dn_dir_clear * nonb_here / nonb_above;
      }
      const double air_ext_t = a.sw.air_ext[(size_t)itransp + (size_t)nspec * il];
      const double trans_dir_clear = exp(-air_ext_t * a.cp.dz[il] / zcos);
      const double int_flux_dir_clear = (air_ext_t > 0.0)
                                            ? flux_dn_dir_clear * (1.0 - trans_dir_clear) * zcos / air_ext_t
                                            : flux_dn_dir_clear * a.cp.dz[il];
      if (own) {
        if ((URBAN ? NREG > 1 : true) && fdir.veg_sunlit_frac && a.cp.veg_ext && a.cp.veg_fraction && a.sw.veg_ssa) {
          const double veg_abs_dir_clear = int_flux_dir_clear * ve * (1.0 - SSB_LAY(a.sw.veg_ssa, g, il)) * vf;
          fdir.veg_sunlit_frac[il] = SSB_FL(fdir, veg_abs_dir, il) / dmax(SSB_EPS, veg_abs_dir_clear);
        }
        if (URBAN && fdir.wall_sunlit_frac)
          fdir.wall_sunlit_frac[il] =
              0.5 * SSB_FL(fdir, wall_in_dir, il) / dmax(SSB_EPS, (f_wall_dir_clear * sin0 * int_flux_dir_clear));
      }
      flux_dn_dir_clear = flux_dn_dir_clear * trans_dir_clear;
    }
  }
  {
    double s_dir = 0.0, dn_d = 0.0, up_d = 0.0, vt_d = 0.0, dn_f = 0.0, up_f = 0.0, vt_f = 0.0;
    SSB_UNROLL
    for (int i = 0; i < d; ++i) s_dir += dir_above[i];
    SSB_UNROLL
    for (int r = 0; r < NREG; ++r) {
      SSB_UNROLL
      for (int js = 0; js < NS; ++js) {
        const int i = js + r * NS;
        dn_d += xa_d[i];
        up_d += ua_d[i];
        vt_d += (xa_d[i] + ua_d[i]) * tang[js] / SSB_PI;
        dn_f += xa_f[i];
        up_f += ua_f[i];
        vt_f += (xa_f[i] + ua_f[i]) * tang[js] / SSB_PI;
      }
    }
    SSB_FC(fdir, ground_dn_dir) = zcos * s_dir;
    SSB_FC(fdir, ground_dn) = zcos * s_dir + dn_d;
    SSB_FC(fdir, ground_net) = SSB_FC(fdir, ground_dn) - up_d;
    SSB_FC(fdir, ground_vertical_diff) = vt_d;
    if (own && fdir.ground_sunlit_frac)
      fdir.ground_sunlit_frac[col] = SSB_FC(fdir, ground_dn_dir) / (zcos * flux_dn_dir_clear);
    SSB_FC(fdif, ground_dn_dir) = 0.0;
    SSB_FC(fdif, ground_dn) = dn_f;
    SSB_FC(fdif, ground_net) = dn_f - up_f;
    SSB_FC(fdif, ground_vertical_diff) = vt_f;
  }
}

// ===========================================================================
// Longwave
// ===========================================================================
template <int NREG, int NS, bool URBAN>
struct LwSweepLayout {
  static constexpr int n = NREG * NS, d = NREG;
  static constexpr int oR = 0, oT = n * n, oIF = 2 * n * n, oSrc = 3 * n * n, oIsrc = oSrc + n, oBook = oIsrc + n;
  static constexpr int oGeo = oBook + 3 * d + 1;  // geometry block (fast_prepare_level)
  static constexpr int oAa = 0, oSa = n * n;
  static constexpr int NRB = URBAN ? NREG + 1 : NREG, m = NRB * NS;
  static constexpr int state_doubles = fast_lw_sweep_elems(n);
  static constexpr int vegNA = NREG > 1 ? n - NS : n, vegI0 = NREG > 1 ? NS : 0;
};

template <int NREG, int NS, bool URBAN>
SSB_HD inline void fast_column_sweeps_lw(const ClassArgs &a, int q, const StateMem &st) {
  typedef LwSweepLayout<NREG, NS, URBAN> Lay;
  constexpr int n = NREG * NS, d = NREG, NRB = URBAN ? NREG + 1 : NREG, m = NRB * NS;
  const SolveCfg &c = a.cfg;
  const int nspec = c.nspec;
  const int ic = q / nspec, g = q % nspec;
  const int col = a.cols[ic];
  const int nlay = a.nlay[col], il1 = layer_index(a, ic, col, 0), ls = layer_step(a);
  const ssb200_canopy_flux &fint = a.f1, &fnorm = a.f2;
  zero_unwritten_lw<NREG, URBAN>(fint, nspec, g, col, il1, nlay, ls);
  zero_unwritten_lw<NREG, URBAN>(fnorm, nspec, g, col, il1, nlay, ls);
  double hw[NS], mu_inv[NS], tang[NS];
  SSB_UNROLL
  for (int js = 0; js < NS; ++js) {
    hw[js] = a.lg.hweight[js];
    mu_inv[js] = 1.0 / a.lg.mu[js];
    tang[js] = a.lg.tan_ang[js];
  }
  const Scr L(a.layer, a.lmax, a.ne_layer, q);
  const Scr W(a.sweep, a.lmax + 1, a.ne_sweep, q);
  const bool full_ua = fint.flux_dn_layer_top != nullptr || fnorm.flux_dn_layer_top != nullptr;
  const double gemis = a.lw.ground_emissivity[(size_t)g + (size_t)nspec * col];
  const double gemission = a.lw.ground_emission[(size_t)g + (size_t)nspec * col];

  // ---- upward sweep: state = [a_above (n x n) | source_above (n)] ------------
  {
    double frac0[3] = {1.0, 0.0, 0.0};
    if (nlay > 0) {
      const bool veg = NREG > 1 || !URBAN;
      region_fractions(c, URBAN ? a.cp.building_fraction[il1] : 0.0,
                       (veg && a.cp.veg_fraction) ? a.cp.veg_fraction[il1] : 0.0, frac0);
    }
    SSB_UNROLL
    for (int i = 0; i < Lay::state_doubles; ++i) st(i) = 0.0;
    SSB_UNROLL
    for (int r = 0; r < NREG; ++r) {
      SSB_UNROLL
      for (int jt = 0; jt < NS; ++jt) {
        SSB_UNROLL
        for (int jf = 0; jf < NS; ++jf) st((jt + r * NS) + n * (jf + r * NS)) = (1.0 - gemis) * hw[jt];
        st(Lay::oSa + jt + r * NS) = (hw[jt] * frac0[r]) * gemission;
      }
    }
  }
  SSB_UNROLL
  for (int i = 0; i < Lay::state_doubles; ++i) W.st(i, 0, st(i));
  for (int jl = 0; jl < nlay; ++jl) {
    const int il = il1 + jl * ls;
    const int seg = (int)L.ld(Lay::oGeo + 7, jl);
    double Ab[n * n], Sb[n];
    if (NREG == 1 || seg == 0)
      lw_up_block<Lay, NREG, NS, n, 0>(st, L, jl, Ab, Sb);
    else if (seg == 1)
      lw_up_block<Lay, NREG, NS, NS, 0>(st, L, jl, Ab, Sb);
    else
      lw_up_block<Lay, NREG, NS, Lay::vegNA, Lay::vegI0>(st, L, jl, Ab, Sb);
    double rb[NS], rs[NS];
    SSB_UNROLL
    for (int js = 0; js < NS; ++js) rb[js] = rs[js] = 0.0;
    if (URBAN) {
      const double bfj = a.cp.building_fraction[il];
      const double exposed = (jl < nlay - 1) ? dmax(0.0, bfj - a.cp.building_fraction[il + ls]) : bfj;
      const double remis = SSB_LAY(a.lw.roof_emissivity, g, il), remission = SSB_LAY(a.lw.roof_emission, g, il);
      SSB_UNROLL
      for (int js = 0; js < NS; ++js) {
        rb[js] = (1.0 - remis) * hw[js];
        rs[js] = hw[js] * remission * exposed;
      }
    }
    double U[12], V[12];
    overlap_above<NREG, URBAN, true>(a, il1, nlay, jl, U, V);
    overlap_matrix<NREG, NRB, NS>(Ab, rb, U, V, st, Lay::oAa);
    SSB_UNROLL
    for (int u = 0; u < NREG; ++u) {
      SSB_UNROLL
      for (int jt = 0; jt < NS; ++jt) {
        double s = 0.0;
        SSB_UNROLL
        for (int lo = 0; lo < NREG; ++lo) s = fma(U[u + NREG * lo], Sb[lo * NS + jt], s);
        if (URBAN) s = fma(U[u + NREG * NREG], rs[jt], s);
        st(Lay::oSa + u * NS + jt) = s;
      }
    }
    if (jl + 1 < nlay) {  // (see the shortwave sweep)
      const int sn = (NREG == 1 || full_ua) ? 0 : (int)L.ld(Lay::oGeo + 7, jl + 1);
      if (sn == 0) {
        SSB_UNROLL
        for (int i = 0; i < Lay::state_doubles; ++i) W.st(i, jl + 1, st(i));
      } else if (sn == 1) {
        interface_store_pruned<Lay, n, NS, 0, 1, 0>(st, W, jl + 1);
      } else {
        interface_store_pruned<Lay, n, Lay::vegNA, Lay::vegI0, 1, 0>(st, W, jl + 1);
      }
    }
  }
  double top_emissivity, top_emission = 0.0;
  {
    double sAll = 0.0;
    SSB_UNROLL
    for (int i = 0; i < NS; ++i) {
      double s = 0.0;
      SSB_UNROLL
      for (int j = 0; j < NS; ++j) s = fma(st(i + n * j), hw[j], s);
      sAll += s;
      top_emission += st(Lay::oSa + i);
    }
    top_emissivity = 1.0 - sAll;
    a.bc.lw_emissivity[(size_t)g + (size_t)nspec * col] = top_emissivity;
    a.bc.lw_emission[(size_t)g + (size_t)nspec * col] = top_emission;
  }

  // ---- downward sweep: internal emission (suffix i) and incoming flux (suffix f) together ----
  double xa_i[n], xa_f[n], ua_i[n], ua_f[n];
  SSB_UNROLL
  for (int i = 0; i < n; ++i) xa_i[i] = xa_f[i] = ua_i[i] = ua_f[i] = 0.0;
  SSB_UNROLL
  for (int js = 0; js < NS; ++js) xa_f[js] = hw[js];
  SSB_FC(fint, top_dn) = 0.0;
  SSB_FC(fint, top_net) = -top_emission;
  SSB_FC(fnorm, top_dn) = 1.0;
  SSB_FC(fnorm, top_net) = top_emissivity;
  for (int jl = nlay - 1; jl >= 0; --jl) {
    const int il = il1 + jl * ls;
    const int seg = (int)L.ld(Lay::oGeo + 7, jl);
    double f_wall[3], od_scaling[3];
    SSB_UNROLL
    for (int r = 0; r < 3; ++r) {
      f_wall[r] = L.ld(Lay::oGeo + r, jl);
      od_scaling[r] = L.ld(Lay::oGeo + 3 + r, jl);
    }
    const bool veg = NREG > 1 || !URBAN;
    const double ve = (veg && a.cp.veg_ext) ? a.cp.veg_ext[il] : 0.0;
    double xb_i[m], xb_f[m];
    {
      double U[12], V[12];
      overlap_above<NREG, URBAN, true>(a, il1, nlay, jl, U, V);
      expand_down<NREG, NRB, NS>(V, xa_i, xb_i);
      expand_down<NREG, NRB, NS>(V, xa_f, xb_f);
    }
    double ub_i[m], ub_f[m], if_i[n], if_f[n];
    if (NREG == 1 || seg == 0)
      lw_down_block<Lay, NREG, NS, n, 0>(L, W, jl, xb_i, xb_f, xa_i, xa_f, ub_i, ub_f, ua_i, ua_f, if_i, if_f);
    else if (seg == 1) {
      if (full_ua || jl == 0)
        lw_down_block<Lay, NREG, NS, NS, 0, true>(L, W, jl, xb_i, xb_f, xa_i, xa_f, ub_i, ub_f, ua_i, ua_f, if_i, if_f);
      else
        lw_down_block<Lay, NREG, NS, NS, 0, false>(L, W, jl, xb_i, xb_f, xa_i, xa_f, ub_i, ub_f, ua_i, ua_f, if_i, if_f);
    } else {
      if (full_ua || jl == 0)
        lw_down_block<Lay, NREG, NS, Lay::vegNA, Lay::vegI0, true>(L, W, jl, xb_i, xb_f, xa_i, xa_f, ub_i, ub_f, ua_i, ua_f,
                                                                  if_i, if_f);
      else
        lw_down_block<Lay, NREG, NS, Lay::vegNA, Lay::vegI0, false>(L, W, jl, xb_i, xb_f, xa_i, xa_f, ub_i, ub_f, ua_i, ua_f,
                                                                   if_i, if_f);
    }
    SSB_UNROLL
    for (int i = n; i < m; ++i) ub_i[i] = ub_f[i] = 0.0;
    if (URBAN) {
      const double bfj = a.cp.building_fraction[il];
      const double exposed = (jl < nlay - 1) ? dmax(0.0, bfj - a.cp.building_fraction[il + ls]) : bfj;
      const double remis = SSB_LAY(a.lw.roof_emissivity, g, il), remission = SSB_LAY(a.lw.roof_emission, g, il);
      double sroof_i = 0.0, sroof_f = 0.0, rup_i = 0.0, rup_f = 0.0;
      SSB_UNROLL
      for (int js = 0; js < NS; ++js) {
        sroof_i += xb_i[n + js];
        sroof_f += xb_f[n + js];
      }
      SSB_UNROLL
      for (int js = 0; js < NS; ++js) {
        ub_i[n + js] = (1.0 - remis) * hw[js] * sroof_i + hw[js] * remission * exposed;
        ub_f[n + js] = (1.0 - remis) * hw[js] * sroof_f;
        rup_i += ub_i[n + js];
        rup_f += ub_f[n + js];
      }
      SSB_FL(fint, roof_in, il) = sroof_i;
      SSB_FL(fint, roof_net, il) = sroof_i - rup_i;
      SSB_FL(fnorm, roof_in, il) = sroof_f;
      SSB_FL(fnorm, roof_net, il) = sroof_f - rup_f;
    }
    if (fint.flux_dn_layer_top || fnorm.flux_dn_layer_top) {
      double s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      SSB_UNROLL
      for (int i = 0; i < n; ++i) {
        s[0] += xb_i[i];
        s[1] += xa_i[i];
        s[2] += ub_i[i];
        s[3] += ua_i[i];
        s[4] += xb_f[i];
        s[5] += xa_f[i];
        s[6] += ub_f[i];
        s[7] += ua_f[i];
      }
      if (fint.flux_dn_layer_top) {
        SSB_FL(fint, flux_dn_layer_top, il) = s[0];
        SSB_FL(fint, flux_dn_layer_base, il) = s[1];
        SSB_FL(fint, flux_up_layer_top, il) = s[2];
        SSB_FL(fint, flux_up_layer_base, il) = s[3];
      }
      if (fnorm.flux_dn_layer_top) {
        SSB_FL(fnorm, flux_dn_layer_top, il) = s[4];
        SSB_FL(fnorm, flux_dn_layer_base, il) = s[5];
        SSB_FL(fnorm, flux_up_layer_top, il) = s[6];
        SSB_FL(fnorm, flux_up_layer_base, il) = s[7];
      }
    }
    double book[3 * d + 1];
    SSB_UNROLL
    for (int i = 0; i < 3 * d + 1; ++i) book[i] = L.ld(Lay::oBook + i, jl);
    double smu_i[NREG], smu_f[NREG], stan_i[NREG], stan_f[NREG];
    SSB_UNROLL
    for (int r = 0; r < NREG; ++r) {
      smu_i[r] = smu_f[r] = stan_i[r] = stan_f[r] = 0.0;
      SSB_UNROLL
      for (int js = 0; js < NS; ++js) {
        smu_i[r] = fma(if_i[r * NS + js], mu_inv[js], smu_i[r]);
        smu_f[r] = fma(if_f[r * NS + js], mu_inv[js], smu_f[r]);
        stan_i[r] = fma(if_i[r * NS + js], tang[js], stan_i[r]);
        stan_f[r] = fma(if_f[r * NS + js], tang[js], stan_f[r]);
      }
    }
    const double dz = a.cp.dz[il];
    const double air_abs = SSB_LAY(a.lw.air_ext, g, il) * (1.0 - SSB_LAY(a.lw.air_ssa, g, il));
    SSB_FL(fint, clear_air_abs, il) = air_abs * smu_i[0] - book[0] * dz;
    SSB_FL(fnorm, clear_air_abs, il) = air_abs * smu_f[0];
    if (NREG > 1) {
      const double vabs = ve * (1.0 - SSB_LAY(a.lw.veg_ssa, g, il));
      double air_i = 0.0, veg_i = 0.0, air_f = 0.0, veg_f = 0.0;
      SSB_UNROLL
      for (int r = 1; r < NREG; ++r) {
        air_i += air_abs * smu_i[r] - book[d + r] * dz;
        veg_i += vabs * smu_i[r] * od_scaling[r] - book[2 * d + r] * dz;
        air_f += air_abs * smu_f[r];
        veg_f += vabs * smu_f[r] * od_scaling[r];
      }
      SSB_FL(fint, veg_air_abs, il) = air_i;
      SSB_FL(fint, veg_abs, il) = veg_i;
      SSB_FL(fnorm, veg_air_abs, il) = air_f;
      SSB_FL(fnorm, veg_abs, il) = veg_f;
    }
    if (URBAN) {
      double win_i = 0.0, win_f = 0.0;
      SSB_UNROLL
      for (int r = 0; r < NREG; ++r) {
        win_i += f_wall[r] * stan_i[r];
        win_f += f_wall[r] * stan_f[r];
      }
      const double wemis = SSB_LAY(a.lw.wall_emissivity, g, il);
      SSB_FL(fint, wall_in, il) = win_i;
      SSB_FL(fint, wall_net, il) = win_i * wemis - book[3 * d] * dz;
      SSB_FL(fnorm, wall_in, il) = win_f;
      SSB_FL(fnorm, wall_net, il) = win_f * wemis;
    }
  }
  {
    double dn_i = 0.0, up_i = 0.0, vt_i = 0.0, dn_f = 0.0, up_f = 0.0, vt_f = 0.0;
    SSB_UNROLL
    for (int r = 0; r < NREG; ++r) {
      SSB_UNROLL
      for (int js = 0; js < NS; ++js) {
        const int i = js + r * NS;
        dn_i += xa_i[i];
        up_i += ua_i[i];
        vt_i += (xa_i[i] + ua_i[i]) * tang[js] / SSB_PI;
        dn_f += xa_f[i];
        up_f += ua_f[i];
        vt_f += (xa_f[i] + ua_f[i]) * tang[js] / SSB_PI;
      }
    }
    SSB_FC(fint, ground_dn) = dn_i;
    SSB_FC(fint, ground_net) = dn_i - up_i;
    SSB_FC(fnorm, ground_dn) = dn_f;
    SSB_FC(fnorm, ground_net) = dn_f - up_f;
    // forest_lw:687-694 accumulates the normalised pass into lw_internal as well
    if (URBAN) {
      SSB_FC(fint, ground_vertical_diff) = vt_i;
      SSB_FC(fnorm, ground_vertical_diff) = vt_f;
    } else {
      SSB_FC(fint, ground_vertical_diff) = vt_i + vt_f;
      SSB_FC(fnorm, ground_vertical_diff) = 0.0;
    }
  }
}

}  // namespace ssb
