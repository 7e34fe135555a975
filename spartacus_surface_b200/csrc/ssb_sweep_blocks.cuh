// ssb_sweep_blocks.cuh - the adding steps of the register-resident sweeps restricted to the block of
// regions a layer actually solves.
//
// A layer without vegetation solves only its clear region, a layer without clear air only its
// vegetated regions (radsurf_urban_sw.F90:512-583): its R, T, S, E and integrated-flux matrices are
// zero outside the block A = [I0, I0 + NA) of stream indices (regions [R0, R0 + DA)).  The interface
// state (a_above, d_above / source_above) stays full size, but with R = [R_AA 0; 0 0]
//     D = I - a_above R = [D_AA 0; D_NA I],  D_AA = I - a_AA R_AA,  D_NA = -a_NA R_AA
// so every solve of the adding method reduces to the order-NA block:
//     (D^-1 w)_A = D_AA^-1 w_A                       whatever w is outside A,
//     D^-1 [r_A; 0] = [x_A; a_NA (R_AA x_A)]         with x_A = D_AA^-1 r_A,
//     a_below = R + T D^-1 a_above T = [R_AA + T_AA D_AA^-1 a_AA T_AA, 0; 0, 0]   (likewise d_below, source_below).
// Half of the layers of the benchmark canopy are clear-only (order 2 instead of 6): with the columns of
// a launch ordered by segment pattern the switch below is uniform per warp, and those layers execute a
// tenth of the arithmetic of a full one instead of multiplying structural zeros.  The LU factors of
// D_AA never go to the interface scratch: the downward step rebuilds them from the a_AA and R_AA it
// loads for its own products (denominator_lu), bit for bit the factors of the upward step.
// Same recurrences as radsurf_urban_sw.F90:603-984 / radsurf_urban_lw.F90:548-858 (and the forest
// equivalents); NA = n, I0 = 0 is the unrestricted step.
#pragma once
#include "ssb_small.cuh"

namespace ssb {

// The interface state stored at level jl is consumed by layer jl alone (downward pass).  A consumer that
// solves only the block A = [I0, I0 + NA) and does not need the upwelling flux outside it reads only the
// rows and columns of a_above that touch A, and the A rows of the vector part of the state: NVC columns
// starting at V0 of d_above (the direct beam of the block's regions) or source_above (NVC = 1).  The rest
// of the state never goes to HBM (a clear-only layer at 2 streams: 22 instead of 54 doubles).
template <class Lay, int n, int NA, int I0, int NVC, int V0, class ScrT>
SSB_HDI void interface_store_pruned(const StateMem &st, const ScrT &W, int lev) {
  SSB_UNROLL
  for (int j = 0; j < n; ++j) {
    SSB_UNROLL
    for (int i = 0; i < n; ++i) {
      if ((i >= I0 && i < I0 + NA) || (j >= I0 && j < I0 + NA)) W.st(Lay::oAa + i + n * j, lev, st(Lay::oAa + i + n * j));
    }
  }
  constexpr int oV = n * n;  // d_above (n x d) or source_above (n) follows a_above in the state
  SSB_UNROLL
  for (int k = 0; k < NVC; ++k) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) W.st(oV + (I0 + i) + n * (V0 + k), lev, st(oV + (I0 + i) + n * (V0 + k)));
  }
}

// ---------------------------------------------------------------------------------------------
// Shortwave
// ---------------------------------------------------------------------------------------------
// upward: Ab (n x n) = a_below street part, Db (n x d) = d_below street part (zeros outside the block)
// D_AA = I - a_AA R_AA factored in place into LU, with the operation order of the upward steps
// (sw_up_block / lw_up_block build the same matrix interleaved with a_AA T_AA): the downward steps
// call this on the same a_AA and R_AA and so solve with exactly the factors of the upward step.
template <int NA>
SSB_HDI void denominator_lu(const double *Aa, const double *Ra, double *LU) {
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) LU[i + NA * j] = (i == j) ? 1.0 : 0.0;
    SSB_UNROLL
    for (int k = 0; k < NA; ++k) {
      SSB_UNROLL
      for (int i = 0; i < NA; ++i) LU[i + NA * j] = fma(-Aa[i + NA * k], Ra[k + NA * j], LU[i + NA * j]);
    }
  }
  sm_lu<NA>(LU);
}

template <class Lay, int NREG, int NS, int NA, int I0, class ScrT>
SSB_HDI void sw_up_block(const StateMem &st, const ScrT &L, int jl, double *Ab, double *Db) {
  constexpr int n = NREG * NS, d = NREG, DA = NA / NS, R0 = I0 / NS;
  double Aa[NA * NA], X[NA * NA], Wd[NA * DA];
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) Aa[i + NA * j] = st(Lay::oAa + (I0 + i) + n * (I0 + j));
  }
  // Wd = (d_above E)_A + a_AA S_dn
  SSB_UNROLL
  for (int j = 0; j < DA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) Wd[i + NA * j] = 0.0;
    SSB_UNROLL
    for (int k = 0; k < DA; ++k) {
      const double e = L.ld(Lay::oE + (R0 + k) + d * (R0 + j), jl);
      SSB_UNROLL
      for (int i = 0; i < NA; ++i) Wd[i + NA * j] = fma(st(Lay::oDa + (I0 + i) + n * (R0 + k)), e, Wd[i + NA * j]);
    }
    SSB_UNROLL
    for (int k = 0; k < NA; ++k) {
      const double w = L.ld(Lay::oSdn + (I0 + k) + n * (R0 + j), jl);
      SSB_UNROLL
      for (int i = 0; i < NA; ++i) Wd[i + NA * j] = fma(Aa[i + NA * k], w, Wd[i + NA * j]);
    }
  }
  {
    double LU[NA * NA];
    SSB_UNROLL
    for (int j = 0; j < NA; ++j) {
      SSB_UNROLL
      for (int i = 0; i < NA; ++i) {
        LU[i + NA * j] = (i == j) ? 1.0 : 0.0;
        X[i + NA * j] = 0.0;
      }
      SSB_UNROLL
      for (int k = 0; k < NA; ++k) {
        const double r = L.ld(Lay::oR + (I0 + k) + n * (I0 + j), jl);
        const double t = L.ld(Lay::oT + (I0 + k) + n * (I0 + j), jl);
        SSB_UNROLL
        for (int i = 0; i < NA; ++i) {
          LU[i + NA * j] = fma(-Aa[i + NA * k], r, LU[i + NA * j]);
          X[i + NA * j] = fma(Aa[i + NA * k], t, X[i + NA * j]);
        }
      }
    }
    sm_lu<NA>(LU);
    sm_lu_solve_left<NA, NA>(LU, X);
    sm_lu_solve_left<NA, DA>(LU, Wd);
  }
  SSB_UNROLL
  for (int i = 0; i < n * n; ++i) Ab[i] = 0.0;
  SSB_UNROLL
  for (int i = 0; i < n * d; ++i) Db[i] = 0.0;
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) Ab[(I0 + i) + n * (I0 + j)] = L.ld(Lay::oR + (I0 + i) + n * (I0 + j), jl);
  }
  SSB_UNROLL
  for (int j = 0; j < DA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) Db[(I0 + i) + n * (R0 + j)] = L.ld(Lay::oSup + (I0 + i) + n * (R0 + j), jl);
  }
  SSB_UNROLL
  for (int k = 0; k < NA; ++k) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) {
      const double t = L.ld(Lay::oT + (I0 + i) + n * (I0 + k), jl);
      SSB_UNROLL
      for (int j = 0; j < NA; ++j) Ab[(I0 + i) + n * (I0 + j)] = fma(t, X[k + NA * j], Ab[(I0 + i) + n * (I0 + j)]);
      SSB_UNROLL
      for (int j = 0; j < DA; ++j) Db[(I0 + i) + n * (R0 + j)] = fma(t, Wd[k + NA * j], Db[(I0 + i) + n * (R0 + j)]);
    }
  }
}

// downward: from the fluxes below the interface above the layer (xb_*: first n entries used, dir_below:
// first d entries) to the fluxes just above the layer base and the integrated fluxes.
// Suffix d: direct-source pass, f: diffuse-source pass.  Every output array is full size (n or d).
template <class Lay, int NREG, int NS, int NA, int I0, bool FULL_UA = true, class ScrT>
SSB_HDI void sw_down_block(const ScrT &L, const ScrT &W, int jl, const double *xb_d, const double *xb_f,
                           const double *dir_below, double *xa_d, double *xa_f, double *dir_above, double *ddir,
                           double *refl, double *ub_d, double *ub_f, double *ua_d, double *ua_f, double *if_d,
                           double *if_f, double *idir) {
  constexpr int n = NREG * NS, d = NREG, DA = NA / NS, R0 = I0 / NS;
  // rows of the interface state outside the block are only needed for the upwelling flux outside the
  // block (flux profiles, ground level): without FULL_UA they are neither stored nor loaded
  // (interface_store_pruned)
  constexpr bool all_rows = (NA == n) || FULL_UA;
  double y_d[NA], y_f[NA], z1_d[NA], z1_f[NA], z2_d[NA], z2_f[NA];
  SSB_UNROLL
  for (int i = 0; i < NA; ++i) y_d[i] = y_f[i] = 0.0;
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) {
      const double t = L.ld(Lay::oT + (I0 + i) + n * (I0 + j), jl);
      y_d[i] = fma(t, xb_d[I0 + j], y_d[i]);
      y_f[i] = fma(t, xb_f[I0 + j], y_f[i]);
    }
  }
  SSB_UNROLL
  for (int j = 0; j < DA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) y_d[i] = fma(L.ld(Lay::oSdn + (I0 + i) + n * (R0 + j), jl), dir_below[R0 + j], y_d[i]);
  }
  // dir_above = E dir_below ; refl = d_above dir_above
  SSB_UNROLL
  for (int i = 0; i < d; ++i) dir_above[i] = 0.0;
  SSB_UNROLL
  for (int j = 0; j < DA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < DA; ++i)
      dir_above[R0 + i] = fma(L.ld(Lay::oE + (R0 + i) + d * (R0 + j), jl), dir_below[R0 + j], dir_above[R0 + i]);
  }
  SSB_UNROLL
  for (int i = 0; i < d; ++i) ddir[i] = dir_below[i] - dir_above[i];
  SSB_UNROLL
  for (int i = 0; i < n; ++i) refl[i] = 0.0;
  SSB_UNROLL
  for (int k = 0; k < DA; ++k) {
    SSB_UNROLL
    for (int i = 0; i < n; ++i) {
      if (all_rows || (i >= I0 && i < I0 + NA))
        refl[i] = fma(W.ld(Lay::oDa + i + n * (R0 + k), jl), dir_above[R0 + k], refl[i]);
    }
  }
  // z1 = D_AA^-1 (a_AA y + refl_A) ; z2 = D_AA^-1 (y + R_AA refl_A) ; ub_A = R_AA xb_A
  SSB_UNROLL
  for (int i = 0; i < NA; ++i) {
    z1_d[i] = refl[I0 + i];
    z1_f[i] = 0.0;
    z2_d[i] = y_d[i];
    z2_f[i] = y_f[i];
  }
  SSB_UNROLL
  for (int i = 0; i < n; ++i) ub_d[i] = ub_f[i] = 0.0;
  double Aa[NA * NA], Ra[NA * NA];
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) {
      const double a = W.ld(Lay::oAa + (I0 + i) + n * (I0 + j), jl);
      const double r = L.ld(Lay::oR + (I0 + i) + n * (I0 + j), jl);
      Aa[i + NA * j] = a;
      Ra[i + NA * j] = r;
      z1_d[i] = fma(a, y_d[j], z1_d[i]);
      z1_f[i] = fma(a, y_f[j], z1_f[i]);
      z2_d[i] = fma(r, refl[I0 + j], z2_d[i]);
      ub_d[I0 + i] = fma(r, xb_d[I0 + j], ub_d[I0 + i]);
      ub_f[I0 + i] = fma(r, xb_f[I0 + j], ub_f[I0 + i]);
    }
  }
  {
    double LU[NA * NA];
    denominator_lu<NA>(Aa, Ra, LU);
    sm_lu_solve_left<NA, 1>(LU, z1_d);
    sm_lu_solve_left<NA, 1>(LU, z1_f);
    sm_lu_solve_left<NA, 1>(LU, z2_d);
    sm_lu_solve_left<NA, 1>(LU, z2_f);
  }
  // up_below (street part) += T_AA z1 + S_up dir_below
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) {
      const double t = L.ld(Lay::oT + (I0 + i) + n * (I0 + j), jl);
      ub_d[I0 + i] = fma(t, z1_d[j], ub_d[I0 + i]);
      ub_f[I0 + i] = fma(t, z1_f[j], ub_f[I0 + i]);
    }
  }
  SSB_UNROLL
  for (int j = 0; j < DA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i)
      ub_d[I0 + i] = fma(L.ld(Lay::oSup + (I0 + i) + n * (R0 + j), jl), dir_below[R0 + j], ub_d[I0 + i]);
  }
  // x_above = [z2 on A ; a_NA (R_AA z2) elsewhere]
  SSB_UNROLL
  for (int i = 0; i < n; ++i) xa_d[i] = xa_f[i] = 0.0;
  SSB_UNROLL
  for (int i = 0; i < NA; ++i) {
    xa_d[I0 + i] = z2_d[i];
    xa_f[I0 + i] = z2_f[i];
  }
  if (NA < n) {
    double t_d[NA], t_f[NA];
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) t_d[i] = t_f[i] = 0.0;
    SSB_UNROLL
    for (int j = 0; j < NA; ++j) {
      SSB_UNROLL
      for (int i = 0; i < NA; ++i) {
        const double r = L.ld(Lay::oR + (I0 + i) + n * (I0 + j), jl);
        t_d[i] = fma(r, z2_d[j], t_d[i]);
        t_f[i] = fma(r, z2_f[j], t_f[i]);
      }
    }
    SSB_UNROLL
    for (int j = 0; j < NA; ++j) {
      SSB_UNROLL
      for (int i = 0; i < n; ++i) {
        if (i < I0 || i >= I0 + NA) {
          const double a = W.ld(Lay::oAa + i + n * (I0 + j), jl);
          xa_d[i] = fma(a, t_d[j], xa_d[i]);
          xa_f[i] = fma(a, t_f[j], xa_f[i]);
        }
      }
    }
  }
  // up_above = a_above x_above + refl
  SSB_UNROLL
  for (int i = 0; i < n; ++i) {
    ua_d[i] = refl[i];
    ua_f[i] = 0.0;
  }
  SSB_UNROLL
  for (int j = 0; j < n; ++j) {
    SSB_UNROLL
    for (int i = 0; i < n; ++i) {
      if (all_rows || (i >= I0 && i < I0 + NA)) {
        const double a = W.ld(Lay::oAa + i + n * j, jl);
        ua_d[i] = fma(a, xa_d[j], ua_d[i]);
        ua_f[i] = fma(a, xa_f[j], ua_f[i]);
      }
    }
  }
  // integrated fluxes across the layer (only the solved regions absorb)
  SSB_UNROLL
  for (int i = 0; i < n; ++i) if_d[i] = if_f[i] = 0.0;
  SSB_UNROLL
  for (int i = 0; i < d; ++i) idir[i] = 0.0;
  {
    double cv_d[NA], cv_f[NA];
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) {
      cv_d[i] = xb_d[I0 + i] - xa_d[I0 + i] - ub_d[I0 + i] + ua_d[I0 + i];
      cv_f[i] = xb_f[I0 + i] - xa_f[I0 + i] - ub_f[I0 + i] + ua_f[I0 + i];
    }
    SSB_UNROLL
    for (int j = 0; j < NA; ++j) {
      SSB_UNROLL
      for (int i = 0; i < NA; ++i) {
        const double v = L.ld(Lay::oIdiff + (I0 + i) + n * (I0 + j), jl);
        if_d[I0 + i] = fma(v, cv_d[j], if_d[I0 + i]);
        if_f[I0 + i] = fma(v, cv_f[j], if_f[I0 + i]);
      }
    }
    SSB_UNROLL
    for (int j = 0; j < DA; ++j) {
      SSB_UNROLL
      for (int i = 0; i < DA; ++i)
        idir[R0 + i] = fma(L.ld(Lay::oIdir + (R0 + i) + d * (R0 + j), jl), ddir[R0 + j], idir[R0 + i]);
      SSB_UNROLL
      for (int i = 0; i < NA; ++i)
        if_d[I0 + i] = fma(L.ld(Lay::oIdd + (I0 + i) + n * (R0 + j), jl), ddir[R0 + j], if_d[I0 + i]);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Longwave (suffix i: internal emission pass, f: incoming-flux pass)
// ---------------------------------------------------------------------------------------------
template <class Lay, int NREG, int NS, int NA, int I0, class ScrT>
SSB_HDI void lw_up_block(const StateMem &st, const ScrT &L, int jl, double *Ab, double *Sb) {
  constexpr int n = NREG * NS;
  double Aa[NA * NA], X[NA * NA], v1[NA], src[NA];
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) Aa[i + NA * j] = st(Lay::oAa + (I0 + i) + n * (I0 + j));
  }
  SSB_UNROLL
  for (int i = 0; i < NA; ++i) {
    src[i] = L.ld(Lay::oSrc + I0 + i, jl);
    v1[i] = st(Lay::oSa + I0 + i);
  }
  SSB_UNROLL
  for (int k = 0; k < NA; ++k) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) v1[i] = fma(Aa[i + NA * k], src[k], v1[i]);
  }
  {
    double LU[NA * NA];
    SSB_UNROLL
    for (int j = 0; j < NA; ++j) {
      SSB_UNROLL
      for (int i = 0; i < NA; ++i) {
        LU[i + NA * j] = (i == j) ? 1.0 : 0.0;
        X[i + NA * j] = 0.0;
      }
      SSB_UNROLL
      for (int k = 0; k < NA; ++k) {
        const double r = L.ld(Lay::oR + (I0 + k) + n * (I0 + j), jl);
        const double t = L.ld(Lay::oT + (I0 + k) + n * (I0 + j), jl);
        SSB_UNROLL
        for (int i = 0; i < NA; ++i) {
          LU[i + NA * j] = fma(-Aa[i + NA * k], r, LU[i + NA * j]);
          X[i + NA * j] = fma(Aa[i + NA * k], t, X[i + NA * j]);
        }
      }
    }
    sm_lu<NA>(LU);
    sm_lu_solve_left<NA, NA>(LU, X);
    sm_lu_solve_left<NA, 1>(LU, v1);
  }
  SSB_UNROLL
  for (int i = 0; i < n * n; ++i) Ab[i] = 0.0;
  SSB_UNROLL
  for (int i = 0; i < n; ++i) Sb[i] = 0.0;
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) Ab[(I0 + i) + n * (I0 + j)] = L.ld(Lay::oR + (I0 + i) + n * (I0 + j), jl);
  }
  SSB_UNROLL
  for (int i = 0; i < NA; ++i) Sb[I0 + i] = src[i];
  SSB_UNROLL
  for (int k = 0; k < NA; ++k) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) {
      const double t = L.ld(Lay::oT + (I0 + i) + n * (I0 + k), jl);
      SSB_UNROLL
      for (int j = 0; j < NA; ++j) Ab[(I0 + i) + n * (I0 + j)] = fma(t, X[k + NA * j], Ab[(I0 + i) + n * (I0 + j)]);
      Sb[I0 + i] = fma(t, v1[k], Sb[I0 + i]);
    }
  }
}

template <class Lay, int NREG, int NS, int NA, int I0, bool FULL_UA = true, class ScrT>
SSB_HDI void lw_down_block(const ScrT &L, const ScrT &W, int jl, const double *xb_i, const double *xb_f, double *xa_i,
                           double *xa_f, double *ub_i, double *ub_f, double *ua_i, double *ua_f, double *if_i,
                           double *if_f) {
  constexpr int n = NREG * NS;
  constexpr bool all_rows = (NA == n) || FULL_UA;  // see sw_down_block
  double src[NA], sa[n], y_i[NA], y_f[NA], z1_i[NA], z1_f[NA], z2_i[NA], z2_f[NA];
  SSB_UNROLL
  for (int i = 0; i < n; ++i) sa[i] = (all_rows || (i >= I0 && i < I0 + NA)) ? W.ld(Lay::oSa + i, jl) : 0.0;
  SSB_UNROLL
  for (int i = 0; i < NA; ++i) {
    src[i] = L.ld(Lay::oSrc + I0 + i, jl);
    y_i[i] = src[i];
    y_f[i] = 0.0;
  }
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) {
      const double t = L.ld(Lay::oT + (I0 + i) + n * (I0 + j), jl);
      y_i[i] = fma(t, xb_i[I0 + j], y_i[i]);
      y_f[i] = fma(t, xb_f[I0 + j], y_f[i]);
    }
  }
  SSB_UNROLL
  for (int i = 0; i < NA; ++i) {
    z1_i[i] = sa[I0 + i];
    z1_f[i] = 0.0;
    z2_i[i] = y_i[i];
    z2_f[i] = y_f[i];
  }
  SSB_UNROLL
  for (int i = 0; i < n; ++i) ub_i[i] = ub_f[i] = 0.0;
  SSB_UNROLL
  for (int i = 0; i < NA; ++i) ub_i[I0 + i] = src[i];
  double Aa[NA * NA], Ra[NA * NA];
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) {
      const double a = W.ld(Lay::oAa + (I0 + i) + n * (I0 + j), jl);
      const double r = L.ld(Lay::oR + (I0 + i) + n * (I0 + j), jl);
      Aa[i + NA * j] = a;
      Ra[i + NA * j] = r;
      z1_i[i] = fma(a, y_i[j], z1_i[i]);
      z1_f[i] = fma(a, y_f[j], z1_f[i]);
      z2_i[i] = fma(r, sa[I0 + j], z2_i[i]);
      ub_i[I0 + i] = fma(r, xb_i[I0 + j], ub_i[I0 + i]);
      ub_f[I0 + i] = fma(r, xb_f[I0 + j], ub_f[I0 + i]);
    }
  }
  {
    double LU[NA * NA];
    denominator_lu<NA>(Aa, Ra, LU);
    sm_lu_solve_left<NA, 1>(LU, z1_i);
    sm_lu_solve_left<NA, 1>(LU, z1_f);
    sm_lu_solve_left<NA, 1>(LU, z2_i);
    sm_lu_solve_left<NA, 1>(LU, z2_f);
  }
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) {
      const double t = L.ld(Lay::oT + (I0 + i) + n * (I0 + j), jl);
      ub_i[I0 + i] = fma(t, z1_i[j], ub_i[I0 + i]);
      ub_f[I0 + i] = fma(t, z1_f[j], ub_f[I0 + i]);
    }
  }
  SSB_UNROLL
  for (int i = 0; i < n; ++i) xa_i[i] = xa_f[i] = 0.0;
  SSB_UNROLL
  for (int i = 0; i < NA; ++i) {
    xa_i[I0 + i] = z2_i[i];
    xa_f[I0 + i] = z2_f[i];
  }
  if (NA < n) {
    double t_i[NA], t_f[NA];
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) t_i[i] = t_f[i] = 0.0;
    SSB_UNROLL
    for (int j = 0; j < NA; ++j) {
      SSB_UNROLL
      for (int i = 0; i < NA; ++i) {
        const double r = L.ld(Lay::oR + (I0 + i) + n * (I0 + j), jl);
        t_i[i] = fma(r, z2_i[j], t_i[i]);
        t_f[i] = fma(r, z2_f[j], t_f[i]);
      }
    }
    SSB_UNROLL
    for (int j = 0; j < NA; ++j) {
      SSB_UNROLL
      for (int i = 0; i < n; ++i) {
        if (i < I0 || i >= I0 + NA) {
          const double a = W.ld(Lay::oAa + i + n * (I0 + j), jl);
          xa_i[i] = fma(a, t_i[j], xa_i[i]);
          xa_f[i] = fma(a, t_f[j], xa_f[i]);
        }
      }
    }
  }
  SSB_UNROLL
  for (int i = 0; i < n; ++i) {
    ua_i[i] = sa[i];
    ua_f[i] = 0.0;
  }
  SSB_UNROLL
  for (int j = 0; j < n; ++j) {
    SSB_UNROLL
    for (int i = 0; i < n; ++i) {
      if (all_rows || (i >= I0 && i < I0 + NA)) {
        const double a = W.ld(Lay::oAa + i + n * j, jl);
        ua_i[i] = fma(a, xa_i[j], ua_i[i]);
        ua_f[i] = fma(a, xa_f[j], ua_f[i]);
      }
    }
  }
  // integrated fluxes: int_flux (dn_below + up_above) + int_flux_source
  SSB_UNROLL
  for (int i = 0; i < n; ++i) if_i[i] = if_f[i] = 0.0;
  SSB_UNROLL
  for (int i = 0; i < NA; ++i) if_i[I0 + i] = L.ld(Lay::oIsrc + I0 + i, jl);
  SSB_UNROLL
  for (int j = 0; j < NA; ++j) {
    const double tv_i = xb_i[I0 + j] + ua_i[I0 + j], tv_f = xb_f[I0 + j] + ua_f[I0 + j];
    SSB_UNROLL
    for (int i = 0; i < NA; ++i) {
      const double v = L.ld(Lay::oIF + (I0 + i) + n * (I0 + j), jl);
      if_i[I0 + i] = fma(v, tv_i, if_i[I0 + i]);
      if_f[I0 + i] = fma(v, tv_f, if_f[I0 + i]);
    }
  }
}

}  // namespace ssb
