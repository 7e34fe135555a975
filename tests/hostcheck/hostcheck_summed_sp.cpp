// hostcheck_summed_sp.cpp - TEST INFRASTRUCTURE: the host check of hostcheck.cpp (the product's solver bodies
// compiled for the host, driven by a serial loop through the same launch plan) plus one export that runs the
// plan with the summing scatter of ssb200_radsurf_fluxes_device_sp.  Built into its own library by
// tests/test_hostcheck_fluxes_sp.py; like hostcheck.cpp it is not a product path.
#include "hostcheck.cpp"

#include <list>

// hostcheck_radsurf_summed with the single-precision storage of ssb200_radsurf_fluxes_device_sp (staged
// route): the per-layer inputs and the per-layer members of sw_flux / lw_flux are staged from and scattered
// into float arrays, converted here from the double arguments (whose values must be floats) and widened back
// into them after the run.  Per-layer inputs whose bit is set in `f64_mask` stay double, as the context
// buffers of the device entry's defaults and emission do: bit i is the i-th member of kCanopyMembers,
// kSwMembers and kLwMembers, in that order.  Each staged array thus takes its own precision within one pass.
extern "C" int hostcheck_radsurf_summed_sp(const ssb200_config *config, const ssb200_canopy_properties *cp,
                                           const ssb200_sw_spectral_properties *sw,
                                           const ssb200_lw_spectral_properties *lw, ssb200_boundary_conds_out *bc,
                                           int32_t istartcol, int32_t iendcol, ssb200_canopy_flux *sw_dir,
                                           ssb200_canopy_flux *sw_diff, ssb200_canopy_flux *lw_int,
                                           ssb200_canopy_flux *lw_norm, ssb200_canopy_flux *sw_flux,
                                           ssb200_canopy_flux *lw_flux, const double *top_sw, const double *top_dir,
                                           const double *top_lw, int64_t budget_doubles, int64_t f64_mask) {
  ssb200_canopy_properties fcp = *cp;
  ssb200_sw_spectral_properties fsw;
  ssb200_lw_spectral_properties flw;
  std::memset(&fsw, 0, sizeof(fsw));
  std::memset(&flw, 0, sizeof(flw));
  if (sw) fsw = *sw;
  if (lw) flw = *lw;
  ssb200_canopy_flux fsum_sw = *sw_flux, fsum_lw = *lw_flux;
  const size_t ntot = (size_t)cp->ntotlay;
  std::list<std::vector<float>> store;
  std::vector<std::pair<double *, std::vector<float> *>> back;
  auto to_float = [&](const double *p, size_t n) {
    store.emplace_back(p, p + n);  // (exact: the values are floats)
    return &store.back();
  };
  ssb::StagePrecision prec;
  prec.f32 = true;
  int bit = 0;
  auto inputs = [&](auto &obj, const auto &table, size_t nspec) {
    for (const auto &m : table) {
      const bool keep = (f64_mask >> bit++) & 1;
      auto &member = obj.*m.ptr;
      if (!member || !m.per_layer) continue;
      if (keep)
        prec.f64.push_back(member);
      else
        member = reinterpret_cast<const double *>(to_float(member, ntot * ssb::member_width(m, nspec))->data());
    }
  };
  inputs(fcp, ssb::kCanopyMembers, 1);
  inputs(fsw, ssb::kSwMembers, (size_t)config->nsw);
  inputs(flw, ssb::kLwMembers, (size_t)config->nlw);
  auto summed = [&](ssb200_canopy_flux &f) {
    for (const ssb::FluxMember &m : ssb::kFluxMembers) {
      double *&member = f.*m.ptr;
      if (!member || !m.per_layer) continue;
      std::vector<float> *v = to_float(member, ntot * ssb::member_width(m, (size_t)f.nspec));
      back.push_back({member, v});
      member = reinterpret_cast<double *>(v->data());
    }
  };
  summed(fsum_sw);
  summed(fsum_lw);
  ssb::CallArgs ca{config, &fcp, sw ? &fsw : nullptr, lw ? &flw : nullptr, bc, sw_dir, sw_diff, lw_int, lw_norm};
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
  disp.precision = prec;
  disp.sum_sw.out = &fsum_sw;
  disp.sum_sw.fa = top_dir;
  disp.sum_sw.fb = top_sw;
  disp.sum_sw.fb_minus = top_dir;
  disp.sum_lw.out = &fsum_lw;
  disp.sum_lw.fb = top_lw;
  rc = disp.run(ca, plan, err);
  if (rc) {
    std::fprintf(stderr, "hostcheck: %s\n", err.c_str());
    return rc;
  }
  for (auto &b : back) std::copy(b.second->begin(), b.second->end(), b.first);
  return be.status;
}
