// hostcheck_summed.cpp - TEST INFRASTRUCTURE: the host check of hostcheck.cpp (the product's solver bodies
// compiled for the host, driven by a serial loop through the same launch plan) plus one export that runs the
// plan with the summing scatter of ssb200_radsurf_fluxes_device.  Built into its own library by
// tests/test_hostcheck_fluxes.py; like hostcheck.cpp it is not a product path.
#include "hostcheck.cpp"

// Serial Dispatcher with the summing scatter of ssb200_radsurf_fluxes_device (staged route, register-resident
// bodies): the per-layer members of sw_flux / lw_flux receive top_dir * sw_dir + (top_sw - top_dir) * sw_diff
// and lw_internal + top_lw * lw_norm straight from the staging.  The normalised objects hold the per-column
// members the sweeps and the surface bodies write in place; their per-layer members only mark which members
// are staged (the caller passes the summed object's arrays there).  Returns -100 when the plan does not take
// the staged route.
extern "C" int hostcheck_radsurf_summed(const ssb200_config *config, const ssb200_canopy_properties *cp,
                                        const ssb200_sw_spectral_properties *sw, const ssb200_lw_spectral_properties *lw,
                                        ssb200_boundary_conds_out *bc, int32_t istartcol, int32_t iendcol,
                                        ssb200_canopy_flux *sw_dir, ssb200_canopy_flux *sw_diff,
                                        ssb200_canopy_flux *lw_int, ssb200_canopy_flux *lw_norm,
                                        ssb200_canopy_flux *sw_flux, ssb200_canopy_flux *lw_flux, const double *top_sw,
                                        const double *top_dir, const double *top_lw, int64_t budget_doubles) {
  ssb::CallArgs ca{config, cp, sw, lw, bc, sw_dir, sw_diff, lw_int, lw_norm};
  std::string err;
  int rc = ssb::validate_call(ca, err);
  int c1 = istartcol > 0 ? istartcol : 1, c2 = iendcol > 0 ? iendcol : cp->ncol;
  if (c2 > cp->ncol) c2 = cp->ncol;
  ssb::Plan plan;
  if (!rc) rc = ssb::build_plan(*config, *cp, c1 - 1, c2 - 1, plan, err);
  if (rc) {
    std::fprintf(stderr, "hostcheck: %s\n", err.c_str());
    return rc;
  }
  HostBackend be;
  be.plan = &plan;
  if (budget_doubles > 0) be.budget = (size_t)budget_doubles;
  be.fast = true;
  ssb::host_generic_jacobi() = false;
  ssb::Dispatcher<HostBackend> disp(be);
  if (!disp.all_layers_staged(ca, plan)) return -100;
  disp.sum_sw.out = sw_flux;
  disp.sum_sw.fa = top_dir;
  disp.sum_sw.fb = top_sw;
  disp.sum_sw.fb_minus = top_dir;
  disp.sum_lw.out = lw_flux;
  disp.sum_lw.fb = top_lw;
  rc = disp.run(ca, plan, err);
  if (rc) {
    std::fprintf(stderr, "hostcheck: %s\n", err.c_str());
    return rc;
  }
  return be.status;
}
