// ssb_driver.hpp - host-side launch plan of one radsurf call.
//
// Replaces the column loop + `select case` of radsurf
// (radsurf/radsurf_interface.F90:105-313): columns are bucketed by solver
// class (forest/urban x number of regions) so that every launch runs one
// uniform kernel; Flat and single-layer urban tiles go to the surface kernel.
// Within a class the columns are processed in chunks sized to the scratch
// budget.  The orchestration is a template over a `Backend` (CUDA in
// ssb_api.cu; a serial host loop in tests/hostcheck) so the same plan code is
// exercised by CPU tests.
#pragma once
#include <algorithm>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "ssb_solver.cuh"
#include "ssb_stage.cuh"

namespace ssb {

// The array members of the ABI structs (include/spartacus_b200.h), in declaration order.  Every entry
// marshals its arrays by looping over these tables, so a member is described once: its extent (per
// column, (nspec, ncol), or per packed layer, (nspec, ntotlay)) and whether it is spectral (nspec values
// per column or layer) or not (one).  Members of ssb200_boundary_conds_out belong to the shortwave
// (width nsw) or the longwave band (width nlw).
template <class S, class P>
struct Member {
  P S::*ptr;
  bool per_layer;
  bool spectral;
  bool lw;  // ssb200_boundary_conds_out: longwave member
};
typedef Member<ssb200_canopy_properties, const double *> CanopyMember;
typedef Member<ssb200_sw_spectral_properties, const double *> SwMember;
typedef Member<ssb200_lw_spectral_properties, const double *> LwMember;
typedef Member<ssb200_boundary_conds_out, double *> BcMember;
typedef Member<ssb200_canopy_flux, double *> FluxMember;

constexpr bool kCol = false, kLay = true, kSpec = true, kOne = false;

inline constexpr CanopyMember kCanopyMembers[] = {
    {&ssb200_canopy_properties::cos_sza, kCol, kOne},
    {&ssb200_canopy_properties::dz, kLay, kOne},
    {&ssb200_canopy_properties::building_fraction, kLay, kOne},
    {&ssb200_canopy_properties::building_scale, kLay, kOne},
    {&ssb200_canopy_properties::veg_fraction, kLay, kOne},
    {&ssb200_canopy_properties::veg_scale, kLay, kOne},
    {&ssb200_canopy_properties::veg_ext, kLay, kOne},
    {&ssb200_canopy_properties::veg_fsd, kLay, kOne},
    {&ssb200_canopy_properties::veg_contact_fraction, kLay, kOne}};
inline constexpr SwMember kSwMembers[] = {
    {&ssb200_sw_spectral_properties::air_ext, kLay, kSpec},
    {&ssb200_sw_spectral_properties::air_ssa, kLay, kSpec},
    {&ssb200_sw_spectral_properties::veg_ssa, kLay, kSpec},
    {&ssb200_sw_spectral_properties::ground_albedo, kCol, kSpec},
    {&ssb200_sw_spectral_properties::roof_albedo, kLay, kSpec},
    {&ssb200_sw_spectral_properties::wall_albedo, kLay, kSpec},
    {&ssb200_sw_spectral_properties::wall_specular_frac, kLay, kSpec},
    {&ssb200_sw_spectral_properties::ground_albedo_dir, kCol, kSpec},
    {&ssb200_sw_spectral_properties::roof_albedo_dir, kLay, kSpec}};
inline constexpr LwMember kLwMembers[] = {
    {&ssb200_lw_spectral_properties::air_ext, kLay, kSpec},
    {&ssb200_lw_spectral_properties::air_ssa, kLay, kSpec},
    {&ssb200_lw_spectral_properties::clear_air_planck, kLay, kSpec},
    {&ssb200_lw_spectral_properties::veg_ssa, kLay, kSpec},
    {&ssb200_lw_spectral_properties::veg_planck, kLay, kSpec},
    {&ssb200_lw_spectral_properties::veg_air_planck, kLay, kSpec},
    {&ssb200_lw_spectral_properties::ground_emissivity, kCol, kSpec},
    {&ssb200_lw_spectral_properties::ground_emission, kCol, kSpec},
    {&ssb200_lw_spectral_properties::roof_emissivity, kLay, kSpec},
    {&ssb200_lw_spectral_properties::wall_emissivity, kLay, kSpec},
    {&ssb200_lw_spectral_properties::roof_emission, kLay, kSpec},
    {&ssb200_lw_spectral_properties::wall_emission, kLay, kSpec}};
inline constexpr BcMember kBcMembers[] = {
    {&ssb200_boundary_conds_out::sw_albedo, kCol, kSpec, false},
    {&ssb200_boundary_conds_out::sw_albedo_dir, kCol, kSpec, false},
    {&ssb200_boundary_conds_out::lw_emissivity, kCol, kSpec, true},
    {&ssb200_boundary_conds_out::lw_emission, kCol, kSpec, true}};
inline constexpr FluxMember kFluxMembers[] = {
    {&ssb200_canopy_flux::ground_dn, kCol, kSpec},
    {&ssb200_canopy_flux::ground_net, kCol, kSpec},
    {&ssb200_canopy_flux::ground_vertical_diff, kCol, kSpec},
    {&ssb200_canopy_flux::top_dn, kCol, kSpec},
    {&ssb200_canopy_flux::top_net, kCol, kSpec},
    {&ssb200_canopy_flux::ground_dn_dir, kCol, kSpec},
    {&ssb200_canopy_flux::top_dn_dir, kCol, kSpec},
    {&ssb200_canopy_flux::ground_sunlit_frac, kCol, kOne},
    {&ssb200_canopy_flux::roof_in, kLay, kSpec},
    {&ssb200_canopy_flux::roof_net, kLay, kSpec},
    {&ssb200_canopy_flux::wall_in, kLay, kSpec},
    {&ssb200_canopy_flux::wall_net, kLay, kSpec},
    {&ssb200_canopy_flux::roof_in_dir, kLay, kSpec},
    {&ssb200_canopy_flux::wall_in_dir, kLay, kSpec},
    {&ssb200_canopy_flux::roof_sunlit_frac, kLay, kOne},
    {&ssb200_canopy_flux::wall_sunlit_frac, kLay, kOne},
    {&ssb200_canopy_flux::clear_air_abs, kLay, kSpec},
    {&ssb200_canopy_flux::veg_abs, kLay, kSpec},
    {&ssb200_canopy_flux::veg_air_abs, kLay, kSpec},
    {&ssb200_canopy_flux::veg_abs_dir, kLay, kSpec},
    {&ssb200_canopy_flux::veg_sunlit_frac, kLay, kOne},
    {&ssb200_canopy_flux::flux_dn_layer_top, kLay, kSpec},
    {&ssb200_canopy_flux::flux_up_layer_top, kLay, kSpec},
    {&ssb200_canopy_flux::flux_dn_layer_base, kLay, kSpec},
    {&ssb200_canopy_flux::flux_up_layer_base, kLay, kSpec},
    {&ssb200_canopy_flux::flux_dn_dir_layer_top, kLay, kSpec},
    {&ssb200_canopy_flux::flux_dn_dir_layer_base, kLay, kSpec}};

// The array members follow the integer header members and fill the rest of the struct: a member added to
// the header without a row above fails here.
#define SSB_TABLE_COVERS(S, first, table) \
  static_assert(offsetof(S, first) + sizeof(table) / sizeof(table[0]) * sizeof(double *) == sizeof(S), #table)
SSB_TABLE_COVERS(ssb200_canopy_properties, cos_sza, kCanopyMembers);
SSB_TABLE_COVERS(ssb200_sw_spectral_properties, air_ext, kSwMembers);
SSB_TABLE_COVERS(ssb200_lw_spectral_properties, air_ext, kLwMembers);
SSB_TABLE_COVERS(ssb200_boundary_conds_out, sw_albedo, kBcMembers);
SSB_TABLE_COVERS(ssb200_canopy_flux, ground_dn, kFluxMembers);
#undef SSB_TABLE_COVERS

// values per column or packed layer of a member of a struct with `nspec` spectral intervals
template <class M>
inline size_t member_width(const M &m, size_t nspec) {
  return m.spectral ? nspec : 1;
}

// Lists the per-layer arrays of a pass and redirects the members of `b` to their level-major staging
// buffers (ssb_stage.cuh), carved from `cursor` (NULL: only count).  Returns doubles per (level, column).
// f32: the members of `b` are the caller's float arrays (ssb200_radsurf_device_sp).
// sum: summing scatter (ssb200_radsurf_fluxes_device): both normalised objects f1 and f2 are still staged
// (the kernels write both), and `out` pairs the staging buffers of each member with that member of *sum.
inline size_t stage_plan(ClassArgs &b, bool lw, size_t per_elem, double *cursor, StageList *in, StageList *out,
                         bool f32 = false, const ssb200_canopy_flux *sum = nullptr) {
  size_t elems = 0;
  // stages `member` (listed in `list` unless NULL); returns its staging buffer
  auto add = [&](StageList *list, double *&member, int ns) -> double * {
    if (!member) return nullptr;
    elems += (size_t)ns;
    if (!cursor) return nullptr;
    double *staged = cursor;
    if (list) {
      list->ref[list->n] = member;
      list->staged[list->n] = cursor;
      list->staged2[list->n] = nullptr;
      list->nspec[list->n] = ns;
      list->f32[list->n] = f32 ? 1 : 0;
      list->sum[list->n] = kSumNone;
      ++list->n;
    }
    member = cursor;
    cursor += (size_t)ns * per_elem;
    return staged;
  };
  // per-layer inputs of the canopy and of the pass's spectral properties
  auto inputs = [&](auto &obj, const auto &table) {
    for (const auto &m : table)
      if (m.per_layer) add(in, const_cast<double *&>(obj.*m.ptr), (int)member_width(m, b.cfg.nspec));
  };
  if (in) in->n = 0;
  if (out) out->n = 0;
  inputs(b.cp, kCanopyMembers);
  if (lw)
    inputs(b.lw, kLwMembers);
  else
    inputs(b.sw, kSwMembers);
  for (const FluxMember &m : kFluxMembers) {
    if (!m.per_layer) continue;
    const int w = (int)member_width(m, b.cfg.nspec);
    if (!sum) {
      add(out, b.f1.*m.ptr, w);
      add(out, b.f2.*m.ptr, w);
      continue;
    }
    double *sa = add(nullptr, b.f1.*m.ptr, w), *sb = add(nullptr, b.f2.*m.ptr, w);
    if (!out || !sa || !sb || !(sum->*m.ptr)) continue;
    out->ref[out->n] = sum->*m.ptr;
    out->staged[out->n] = sa;
    out->staged2[out->n] = sb;
    out->nspec[out->n] = w;
    out->f32[out->n] = 0;
    out->sum[out->n] = m.spectral ? kSumScaled : kSumPlain;
    ++out->n;
  }
  return elems;
}

struct ColumnClass {
  int urban, nreg;
  std::vector<int> cols;
};

struct Plan {
  // host copies used to detect a change of the column description between calls
  std::vector<int> nlay, istartlay, irep;
  int c1 = 0, c2 = -1;  // 0-based inclusive range
  int nveg_forest = -1, nveg_urban = -1;
  std::vector<ColumnClass> classes;
  std::vector<int> surface_cols;
  std::vector<int> all_cols;  // concatenation uploaded to the device
  bool valid = false;
  long generation = 0;  // bumped on every rebuild (device copies are refreshed when it changes)
  const int *host_cols(size_t offset) const { return all_cols.data() + offset; }
};

inline int stream_capacity(int ns) {
  if (ns <= 1) return 1;
  if (ns <= 2) return 2;
  if (ns <= 4) return 4;
  if (ns <= 8) return 8;
  return 0;
}

inline LgTable make_lg(const ssb200_legendre_gauss &s) {
  LgTable t;
  std::memset(&t, 0, sizeof(t));
  t.ns = s.nstream;
  for (int i = 0; i < SSB200_MAX_NSTREAM; ++i) {
    t.mu[i] = s.mu[i];
    t.tan_ang[i] = s.tan_ang[i];
    t.weight[i] = s.weight[i];
    t.hweight[i] = s.hweight[i];
    t.vweight[i] = s.vweight[i];
  }
  t.vadjustment = s.vadjustment;
  t.vadjustment2 = s.vadjustment2;
  return t;
}

// Returns 0 or a negative SSB200_ERR_* code; `err` receives the message.
inline int build_plan(const ssb200_config &cfg, const ssb200_canopy_properties &cp, int c1, int c2, Plan &plan,
                      std::string &err) {
  const int ncol = cp.ncol;
  const bool same = plan.valid && plan.c1 == c1 && plan.c2 == c2 && (int)plan.nlay.size() == ncol &&
                    plan.nveg_forest == cfg.n_vegetation_region_forest &&
                    plan.nveg_urban == cfg.n_vegetation_region_urban &&
                    std::memcmp(plan.nlay.data(), cp.nlay, sizeof(int) * ncol) == 0 &&
                    std::memcmp(plan.istartlay.data(), cp.istartlay, sizeof(int) * ncol) == 0 &&
                    std::memcmp(plan.irep.data(), cp.i_representation, sizeof(int) * ncol) == 0;
  if (same) return 0;
  const long generation = plan.generation + 1;
  plan = Plan();
  plan.generation = generation;
  plan.nlay.assign(cp.nlay, cp.nlay + ncol);
  plan.istartlay.assign(cp.istartlay, cp.istartlay + ncol);
  plan.irep.assign(cp.i_representation, cp.i_representation + ncol);
  plan.c1 = c1;
  plan.c2 = c2;
  plan.nveg_forest = cfg.n_vegetation_region_forest;
  plan.nveg_urban = cfg.n_vegetation_region_urban;
  auto class_of = [&](int urban, int nreg) -> ColumnClass & {
    for (auto &k : plan.classes)
      if (k.urban == urban && k.nreg == nreg) return k;
    plan.classes.push_back(ColumnClass{urban, nreg, {}});
    return plan.classes.back();
  };
  for (int j = c1; j <= c2; ++j) {
    const int irep = cp.i_representation[j];
    const int nl = cp.nlay[j];
    if (irep != SSB200_TILE_FLAT) {
      if (nl < 0 || cp.istartlay[j] < 1 || cp.istartlay[j] - 1 + nl > cp.ntotlay) {
        err = "column " + std::to_string(j + 1) + ": layer range outside 1..ntotlay";
        return SSB200_ERR_SHAPE;
      }
    }
    switch (irep) {
      case SSB200_TILE_FLAT:
        plan.surface_cols.push_back(j);
        break;
      case SSB200_TILE_FOREST:
        class_of(0, cfg.n_vegetation_region_forest + 1).cols.push_back(j);
        break;
      case SSB200_TILE_URBAN:
        class_of(1, 1).cols.push_back(j);
        break;
      case SSB200_TILE_VEGETATED_URBAN:
        class_of(1, cfg.n_vegetation_region_urban + 1).cols.push_back(j);
        break;
      case SSB200_TILE_SIMPLE_URBAN:
      case SSB200_TILE_INFINITE_STREET:
        if (nl > 1) {
          err = "Attempt to use simple urban representation with more than one layer";
          return SSB200_ERR_SIMPLE_URBAN_LAYERS;
        }
        plan.surface_cols.push_back(j);
        break;
      default:
        // the reference's select case would skip the column; a code outside the six tile types is
        // an input error, and reporting it keeps stale staging data from reaching the caller
        err = "column " + std::to_string(j + 1) + ": unknown i_representation " + std::to_string(irep);
        return SSB200_ERR_ARG;
    }
  }
  for (auto &k : plan.classes) {
    if (k.nreg < 1 || k.nreg > SSB200_MAX_NREG) {
      err = "number of regions outside 1..3";
      return SSB200_ERR_UNSUPPORTED;
    }
    if (k.nreg > 1 && !cfg.do_vegetation) {
      err = "Attempt to perform radiative transfer with more than one region when vegetation not enabled";
      return SSB200_ERR_ARG;
    }
  }
  for (auto &k : plan.classes) plan.all_cols.insert(plan.all_cols.end(), k.cols.begin(), k.cols.end());
  plan.all_cols.insert(plan.all_cols.end(), plan.surface_cols.begin(), plan.surface_cols.end());
  plan.valid = true;
  return 0;
}

struct CallArgs {
  const ssb200_config *config;
  const ssb200_canopy_properties *cp;  // index arrays on host, doubles on device
  const ssb200_sw_spectral_properties *sw;
  const ssb200_lw_spectral_properties *lw;
  ssb200_boundary_conds_out *bc;
  ssb200_canopy_flux *sw_dir, *sw_diff, *lw_int, *lw_norm;
};

// Backend concept:
//   const int *dev_cols(const Plan&, size_t offset)  device copy of plan.all_cols (+offset)
//   const int *order_chunk(const ClassArgs&, const int *host_cols)   a.cols, possibly reordered
//   const int *dev_nlay(), *dev_istartlay(), *dev_irep()
//   double *scratch(size_t doubles)                  grow-only scratch
//   size_t scratch_budget_doubles()
//   int *dev_status()
//   template<int NS> void layer_sw/layer_lw(const ClassArgs&, long nthreads)
//   template<int NS> void sweeps_sw/sweeps_lw(const ClassArgs&, long nthreads)
//   void surface(const SurfaceArgs&, int nsw_threads, int nlw_threads)
//   bool fused_shape(const SolveCfg&, bool lw, int *private_elems, int *op_elems, int *geo_first)
//        false: no column-resident kernel for this shape (or disabled): split path
//   int fused_slots()                                private tiles (= resident thread blocks)
//   int fused_flags()                                ClassArgs::fused (bit 0 set; bit 1: block-aligned phases)
//   void fused_run(const ClassArgs&, bool lw, long width)
//   bool records_shape(const SolveCfg&, bool lw, int *op_elems)   record sweeps available and enabled
//   void records_run(const ClassArgs&, bool lw, long width)
//   void fork_passes(), begin_pass(bool lw), end_passes()   optional concurrency of the SW and LW passes
//   bool stage_supported(const SolveCfg&)            level-major staging of per-layer arrays enabled for this class
//   void stage(const StageArgs&, bool scatter, bool lw)   gather (inputs -> staging) / scatter (staging -> outputs)
template <class Backend>
struct Dispatcher {
  Backend &be;
  // optional window of global column indices [col_lo, col_hi): lets the host entry
  // pipeline transfers and kernels over blocks of columns without rebuilding the plan
  int col_lo = 0, col_hi = 0x7fffffff;
  // the per-layer members of the call are the caller's float arrays, read and written through the
  // level-major staging only (ssb200_radsurf_device_sp; see all_layers_staged)
  bool f32_layers = false;
  // summing scatter of each pass (ssb200_radsurf_fluxes_device; only valid when all_layers_staged holds):
  // the per-layer members of f1 and f2 exist in the staging buffers of a chunk only, and the scatter
  // writes their scaled sum into `out`.  The per-column members are left to the caller.
  struct PassSum {
    const ssb200_canopy_flux *out = nullptr;  // NULL: plain scatter into f1 and f2
    const double *fa = nullptr, *fb = nullptr, *fb_minus = nullptr;
  };
  PassSum sum_sw, sum_lw;
  explicit Dispatcher(Backend &b) : be(b) {}

  static SolveCfg class_cfg(const ssb200_config &cfg, const ColumnClass &k, bool lw) {
    const ssb200_legendre_gauss &lgs =
        lw ? (k.urban ? cfg.lg_lw_urban : cfg.lg_lw_forest) : (k.urban ? cfg.lg_sw_urban : cfg.lg_sw_forest);
    SolveCfg c;
    std::memset(&c, 0, sizeof(c));
    c.urban = k.urban;
    c.lw = lw ? 1 : 0;
    c.nreg = k.nreg;
    c.ns = lgs.nstream;
    c.nspec = lw ? cfg.nlw : cfg.nsw;
    c.symmetric_scale = k.urban ? cfg.use_symmetric_vegetation_scale_urban : cfg.use_symmetric_vegetation_scale_forest;
    c.isolation = k.urban ? cfg.vegetation_isolation_factor_urban : cfg.vegetation_isolation_factor_forest;
    c.min_veg = cfg.min_vegetation_fraction;
    c.min_bld = cfg.min_building_fraction;
    return c;
  }

  // True when every read and write of a per-layer member in the plan goes through the level-major
  // staging: each class and pass is staged (no column-resident kernels, no unstaged split kernels) and
  // no single-layer urban column is present (the surface kernel reads and writes its layer in place).
  bool all_layers_staged(const CallArgs &ca, const Plan &plan) {
    const ssb200_config &cfg = *ca.config;
    for (int j : plan.surface_cols)
      if (plan.irep[j] == SSB200_TILE_SIMPLE_URBAN || plan.irep[j] == SSB200_TILE_INFINITE_STREET) return false;
    for (const ColumnClass &k : plan.classes)
      for (int pass = 0; pass < 2; ++pass) {
        const bool lw = (pass == 1);
        if (k.cols.empty() || (lw ? !cfg.do_lw : !cfg.do_sw)) continue;
        const SolveCfg c = class_cfg(cfg, k, lw);
        int pe = 0, oe = 0, geo = 0;
        if (be.fused_shape(c, lw, &pe, &oe, &geo) || !be.stage_supported(c)) return false;
      }
    return true;
  }

  template <int NS>
  void run_class(ClassArgs a, bool lw, const Plan &plan, const ColumnClass &k, size_t col_offset) {
    const SolveCfg &c = a.cfg;
    const int n = c.nreg * c.ns, d = c.nreg, nrb = c.urban ? c.nreg + 1 : c.nreg, m = nrb * c.ns;
    const size_t el = lw ? lw_layer_elems(n, c.nreg) : sw_layer_elems(n, d);
    const size_t budget = be.scratch_budget_doubles();
    // column-resident path where the backend has it (1 and 2 streams): one private tile per
    // resident thread block plus one operator record per (problem, level)
    int f_private = 0, f_op = 0, f_geo = 0;
    const bool fused = be.fused_shape(c, lw, &f_private, &f_op, &f_geo);
    const size_t f_tiles = fused ? (size_t)be.fused_slots() * (size_t)f_private * kScratchTile : 0;
    // record sweeps: the split layer kernels, then an upward pass that turns every layer into its
    // down-pass operator record and a downward pass through the records (ssb_fused.cuh MODE 1 / 2)
    int r_op = 0;
    const bool rec = !fused && be.records_shape(c, lw, &r_op);
    // level-major staging of the per-layer arrays (ssb_stage.cuh): register-resident kernels only
    const bool stage = !fused && be.stage_supported(c);
    // interface scratch per level: staged arrays are read by the register-resident sweeps alone (the
    // generic ones refuse them), which keep only a_above and d_above / source_above.  This holds because
    // every shape stage_supported() accepts has a register-resident sweep kernel; should one ever lack
    // it, the backend refuses the generic sweeps on the smaller area instead of overrunning it.
    const size_t es = stage ? (size_t)(lw ? fast_lw_sweep_elems(n) : fast_sw_sweep_elems(n, d))
                            : (size_t)(lw ? lw_sweep_elems(n, m, c.nreg, nrb) : sw_sweep_elems(n, d, m, nrb, c.nreg, nrb));
    size_t stage_elems = 0;
    if (stage) {
      ClassArgs probe = a;
      stage_elems = stage_plan(probe, lw, 0, nullptr, nullptr, nullptr);
    }
    // class columns are ascending: restrict to the window by binary search
    size_t pos = (size_t)(std::lower_bound(k.cols.begin(), k.cols.end(), col_lo) - k.cols.begin());
    const size_t ntot = (size_t)(std::lower_bound(k.cols.begin(), k.cols.end(), col_hi) - k.cols.begin());
    auto need_of = [&](size_t lm, size_t wd) {
      const size_t staging = stage_elems * lm * (wd / (size_t)c.nspec);
      if (rec) return scratch_doubles(el, lm, wd) + scratch_doubles((size_t)r_op, lm > 0 ? lm : 1, wd) + staging;
      return fused ? f_tiles + scratch_doubles((size_t)f_op, lm > 0 ? lm : 1, wd)
                   : scratch_doubles(el, lm, wd) + scratch_doubles(es, lm + 1, wd) + staging;
    };
    while (pos < ntot) {
      // grow the chunk while its scratch (sized by the tallest column) fits the budget
      int lmax = 0;
      size_t cnt = 0;
      while (pos + cnt < ntot) {
        const int nl = plan.nlay[k.cols[pos + cnt]];
        const int lm = std::max(lmax, nl);
        const size_t wd = (cnt + 1) * (size_t)c.nspec;
        if (need_of((size_t)lm, wd) > budget && cnt > 0) break;
        lmax = lm;
        ++cnt;
      }
      a.ncols = (int)cnt;
      a.lmax = lmax;
      a.cols = be.dev_cols(plan, col_offset + pos);
      // the backend may reorder the columns of the chunk (every problem is independent; scratch
      // positions follow the order of a.cols, global arrays are addressed through it)
      a.fused = fused ? be.fused_flags() : 0;
      a.cols = be.order_chunk(a, plan.host_cols(col_offset + pos));
      const size_t width = cnt * (size_t)c.nspec;
      double *s = be.scratch(need_of((size_t)lmax, width));
      if (fused) {
        a.layer = s;
        a.sweep = s + f_tiles;
        a.lmax = lmax > 0 ? lmax : 1;
        a.ne_layer = f_private;
        a.ne_layer_geo = f_geo;
        a.ne_sweep = f_op;
        a.save_profile = (a.f1.flux_dn_layer_top || a.f2.flux_dn_layer_top) ? 1 : 0;
        be.fused_run(a, lw, (long)width);
        pos += cnt;
        continue;
      }
      a.layer = s;
      a.sweep = s + scratch_doubles(el, (size_t)lmax, width);
      a.ne_layer = (int)el;
      a.ne_layer_geo = (int)el - kGeoElems;
      a.ne_sweep = rec ? r_op : (int)es;
      a.save_profile = (a.f1.flux_dn_layer_top || a.f2.flux_dn_layer_top) ? 1 : 0;
      // b: what the kernels see - the caller's arrays, or (staged) the chunk's level-major copies
      ClassArgs b = a;
      StageArgs sin, sout;
      const bool staged = stage && lmax > 0;
      if (staged) {
        double *cursor = a.sweep + (rec ? scratch_doubles((size_t)r_op, (size_t)lmax, width)
                                        : scratch_doubles(es, (size_t)lmax + 1, width));
        const PassSum &ps = lw ? sum_lw : sum_sw;
        stage_plan(b, lw, (size_t)lmax * cnt, cursor, &sin.list, &sout.list, f32_layers, ps.out);
        sin.fa = sin.fb = sin.fb_minus = nullptr;
        sout.fa = ps.fa;
        sout.fb = ps.fb;
        sout.fb_minus = ps.fb_minus;
        b.lstride = (int)cnt;
        sin.cols = sout.cols = a.cols;
        sin.nlay = sout.nlay = a.nlay;
        sin.istartlay = sout.istartlay = a.istartlay;
        sin.ncols = sout.ncols = (int)cnt;
        sin.lmax = sout.lmax = lmax;
        be.stage(sin, false, lw);
      }
      if (lmax > 0) {
        if (lw)
          be.template layer_lw<NS>(b, (long)width * lmax);
        else
          be.template layer_sw<NS>(b, (long)width * lmax);
      }
      if (rec)
        be.records_run(b, lw, (long)width);
      else if (lw)
        be.template sweeps_lw<NS>(b, (long)width);
      else
        be.template sweeps_sw<NS>(b, (long)width);
      if (staged) be.stage(sout, true, lw);
      pos += cnt;
    }
  }

  int run(const CallArgs &ca, const Plan &plan, std::string &err) {
    const ssb200_config &cfg = *ca.config;
    size_t col_offset = 0;
    // the shortwave and the longwave pass of a class are independent (disjoint outputs, read-only
    // inputs): the backend may run them on two streams with separate scratch (begin_pass / end_passes)
    be.fork_passes();
    for (const ColumnClass &k : plan.classes) {
      for (int pass = 0; pass < 2; ++pass) {
        const bool lw = (pass == 1);
        if (lw ? !cfg.do_lw : !cfg.do_sw) continue;
        be.begin_pass(lw);
        const ssb200_legendre_gauss &lgs =
            lw ? (k.urban ? cfg.lg_lw_urban : cfg.lg_lw_forest) : (k.urban ? cfg.lg_sw_urban : cfg.lg_sw_forest);
        const int cap = stream_capacity(lgs.nstream);
        if (lgs.nstream < 1 || cap == 0) {
          err = "number of streams outside 1..8";
          return SSB200_ERR_UNSUPPORTED;
        }
        ClassArgs a;
        std::memset(&a, 0, sizeof(a));
        a.cfg = class_cfg(cfg, k, lw);
        a.lg = make_lg(lgs);
        a.nlay = be.dev_nlay();
        a.istartlay = be.dev_istartlay();
        a.cp = *ca.cp;
        if (lw) {
          a.lw = *ca.lw;
          a.f1 = *ca.lw_int;
          a.f2 = *ca.lw_norm;
        } else {
          a.sw = *ca.sw;
          a.f1 = *ca.sw_dir;
          a.f2 = *ca.sw_diff;
        }
        a.use_sw_direct_albedo = cfg.use_sw_direct_albedo;
        a.bc = *ca.bc;
        a.status = be.dev_status();
        switch (cap) {
          case 1: run_class<1>(a, lw, plan, k, col_offset); break;
          case 2: run_class<2>(a, lw, plan, k, col_offset); break;
          case 4: run_class<4>(a, lw, plan, k, col_offset); break;
          default: run_class<8>(a, lw, plan, k, col_offset); break;
        }
      }
      col_offset += k.cols.size();
    }
    be.end_passes();
    const size_t s_lo = (size_t)(std::lower_bound(plan.surface_cols.begin(), plan.surface_cols.end(), col_lo) -
                                 plan.surface_cols.begin());
    const size_t s_hi = (size_t)(std::lower_bound(plan.surface_cols.begin(), plan.surface_cols.end(), col_hi) -
                                 plan.surface_cols.begin());
    if (s_hi > s_lo) {
      SurfaceArgs s;
      std::memset(&s, 0, sizeof(s));
      s.ncols = (int)(s_hi - s_lo);
      s.nsw = cfg.nsw;
      s.nlw = cfg.nlw;
      s.do_sw = cfg.do_sw;
      s.do_lw = cfg.do_lw;
      s.use_sw_direct_albedo = cfg.use_sw_direct_albedo;
      s.min_veg = cfg.min_vegetation_fraction;
      s.min_bld = cfg.min_building_fraction;
      s.cols = be.dev_cols(plan, col_offset + s_lo);
      s.nlay = be.dev_nlay();
      s.istartlay = be.dev_istartlay();
      s.irep = be.dev_irep();
      s.cp = *ca.cp;
      if (cfg.do_sw) {
        s.sw = *ca.sw;
        s.sw_dir = *ca.sw_dir;
        s.sw_diff = *ca.sw_diff;
      }
      if (cfg.do_lw) {
        s.lw = *ca.lw;
        s.lw_int = *ca.lw_int;
        s.lw_norm = *ca.lw_norm;
      }
      s.bc = *ca.bc;
      be.surface(s, cfg.do_sw ? s.ncols * cfg.nsw : 0, cfg.do_lw ? s.ncols * cfg.nlw : 0);
    }
    return 0;
  }
};

// Argument checks shared by both entry points; returns 0 or SSB200_ERR_*.
inline int validate_call(const CallArgs &ca, std::string &err) {
  if (!ca.config || !ca.cp || !ca.bc) {
    err = "config, canopy_props and bc_out must not be NULL";
    return SSB200_ERR_ARG;
  }
  const ssb200_config &cfg = *ca.config;
  const ssb200_canopy_properties &cp = *ca.cp;
  if (cp.ncol < 0 || !cp.nlay || !cp.istartlay || !cp.i_representation) {
    err = "canopy_props: nlay/istartlay/i_representation missing";
    return SSB200_ERR_ARG;
  }
  if (cfg.do_sw) {
    if (!ca.sw || !ca.sw_dir || !ca.sw_diff || !cp.cos_sza || !ca.bc->sw_albedo || !ca.bc->sw_albedo_dir) {
      err = "do_sw requires sw_spectral_props, cos_sza, sw_norm_dir, sw_norm_diff and bc_out%sw_albedo*";
      return SSB200_ERR_ARG;
    }
    if (ca.sw->nspec != cfg.nsw || ca.sw_dir->nspec != cfg.nsw || ca.sw_diff->nspec != cfg.nsw) {
      err = "shortwave spectral resolution mismatch (config%nsw vs arrays)";
      return SSB200_ERR_SHAPE;
    }
    if (cfg.use_sw_direct_albedo && !ca.sw->ground_albedo_dir) {
      err = "use_sw_direct_albedo set but ground_albedo_dir not allocated";
      return SSB200_ERR_ARG;
    }
  }
  if (cfg.do_lw) {
    if (!ca.lw || !ca.lw_int || !ca.lw_norm || !ca.bc->lw_emissivity || !ca.bc->lw_emission) {
      err = "do_lw requires lw_spectral_props, lw_internal, lw_norm and bc_out%lw_*";
      return SSB200_ERR_ARG;
    }
    if (ca.lw->nspec != cfg.nlw || ca.lw_int->nspec != cfg.nlw || ca.lw_norm->nspec != cfg.nlw) {
      err = "longwave spectral resolution mismatch (config%nlw vs arrays)";
      return SSB200_ERR_SHAPE;
    }
  }
  return 0;
}

// The members each tile class present in the plan dereferences (the kernels do not test them):
// a NULL one is an argument error here instead of an illegal address on the device, which would
// poison the CUDA context of the whole process.
inline int validate_members(const CallArgs &ca, const Plan &plan, std::string &err) {
  const ssb200_config &cfg = *ca.config;
  const ssb200_canopy_properties &cp = *ca.cp;
  bool layered = false, urban = false, veg = false, three = false, simple = false;
  for (const auto &k : plan.classes) {
    if (k.cols.empty()) continue;
    layered = true;
    urban = urban || k.urban;
    veg = veg || k.nreg > 1 || !k.urban;
    three = three || k.nreg == 3;
  }
  for (int j : plan.surface_cols) simple = simple || plan.irep[j] >= SSB200_TILE_SIMPLE_URBAN;
  std::string missing;
  auto need = [&](const void *p, const char *name) {
    if (!p) missing += (missing.empty() ? "" : ", ") + std::string(name);
  };
  if (layered || simple) need(cp.dz, "canopy_props%dz");
  if (urban || simple) {
    need(cp.building_fraction, "canopy_props%building_fraction");
    need(cp.building_scale, "canopy_props%building_scale");
  }
  if (veg) {
    need(cp.veg_fraction, "canopy_props%veg_fraction");
    need(cp.veg_scale, "canopy_props%veg_scale");
    need(cp.veg_ext, "canopy_props%veg_ext");
  }
  if (three) need(cp.veg_fsd, "canopy_props%veg_fsd");
  if (cfg.do_sw) {
    const ssb200_sw_spectral_properties &sw = *ca.sw;
    need(sw.ground_albedo, "sw%ground_albedo");
    if (layered) {
      need(sw.air_ext, "sw%air_ext");
      need(sw.air_ssa, "sw%air_ssa");
    }
    if (veg) need(sw.veg_ssa, "sw%veg_ssa");
    if (urban || simple) {
      need(sw.roof_albedo, "sw%roof_albedo");
      need(sw.wall_albedo, "sw%wall_albedo");
    }
    if (urban) need(sw.wall_specular_frac, "sw%wall_specular_frac");
  }
  if (cfg.do_lw) {
    const ssb200_lw_spectral_properties &lw = *ca.lw;
    need(lw.ground_emissivity, "lw%ground_emissivity");
    need(lw.ground_emission, "lw%ground_emission");
    if (layered) {
      need(lw.air_ext, "lw%air_ext");
      need(lw.air_ssa, "lw%air_ssa");
      need(lw.clear_air_planck, "lw%clear_air_planck");
    }
    if (veg) {
      need(lw.veg_ssa, "lw%veg_ssa");
      need(lw.veg_planck, "lw%veg_planck");
      need(lw.veg_air_planck, "lw%veg_air_planck");
    }
    if (urban || simple) {
      need(lw.roof_emissivity, "lw%roof_emissivity");
      need(lw.wall_emissivity, "lw%wall_emissivity");
      need(lw.roof_emission, "lw%roof_emission");
      need(lw.wall_emission, "lw%wall_emission");
    }
  }
  if (!missing.empty()) {
    err = "members needed by the tile types present are not allocated: " + missing;
    return SSB200_ERR_ARG;
  }
  return 0;
}

}  // namespace ssb
