/* spartacus_b200.h - C ABI of the B200-native SPARTACUS-Surface solver path.
 *
 * This is the drop-in boundary for ONE path of ecmwf/spartacus-surface: the
 * body of `radsurf` (reference radsurf/radsurf_interface.F90:20-317) and
 * everything it calls.  The reference has no FFI; its seam is the Fortran
 * module procedure `radsurf_interface::radsurf`.  A Fortran ISO_C_BINDING shim
 * (spartacus_surface_b200/fortran/radsurf_interface_b200.F90) takes c_loc()
 * of every allocated member of the reference derived types and calls
 * ssb200_radsurf().  The structs below therefore mirror those derived types
 * member by member; all arrays keep the reference layout:
 *   column-major, spectral index fastest, (nspec, ncol) or packed ragged
 *   (nspec, ntotlay) with 1-based `istartlay`.
 * A NULL pointer means "member not allocated" in the Fortran sense.
 *
 * The same structs are consumed by the CPU oracle (oracle/), which is test
 * infrastructure only and is never linked into the product library.
 */
#ifndef SPARTACUS_B200_H
#define SPARTACUS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSB200_MAX_NSTREAM 16
#define SSB200_MAX_NREG 3

/* Tile representation codes: radsurf/radsurf_canopy_properties.F90:26-33 */
enum {
  SSB200_TILE_FLAT = 0,
  SSB200_TILE_FOREST = 1,
  SSB200_TILE_URBAN = 2,
  SSB200_TILE_VEGETATED_URBAN = 3,
  SSB200_TILE_SIMPLE_URBAN = 4,
  SSB200_TILE_INFINITE_STREET = 5
};

/* Return codes.  >0 from ssb200_radsurf*: number of (column, interval)
 * problems flagged non-finite / non-converged (reference would have trapped an
 * FP exception, Makefile_include.gfortran:28). */
enum {
  SSB200_OK = 0,
  SSB200_ERR_ARG = -1,        /* NULL / inconsistent argument */
  SSB200_ERR_SHAPE = -2,      /* spectral/shape mismatch */
  SSB200_ERR_UNSUPPORTED = -3,/* nreg/nstream outside compiled range */
  SSB200_ERR_CUDA = -4,       /* CUDA runtime failure (see ssb200_last_error) */
  SSB200_ERR_NOGPU = -5,      /* no CUDA device: there is NO CPU fallback */
  SSB200_ERR_SIMPLE_URBAN_LAYERS = -6 /* radsurf_interface.F90:281-284 */
};

/* legendre_gauss_type: radtool/radtool_legendre_gauss.F90:25-48 */
typedef struct ssb200_legendre_gauss {
  int32_t nstream;
  int32_t pad_;
  double mu[SSB200_MAX_NSTREAM];
  double sin_ang[SSB200_MAX_NSTREAM];
  double tan_ang[SSB200_MAX_NSTREAM];
  double weight[SSB200_MAX_NSTREAM];
  double hweight[SSB200_MAX_NSTREAM];
  double vweight[SSB200_MAX_NSTREAM];
  double vadjustment;
  double vadjustment2;
} ssb200_legendre_gauss;

/* config_type members read under radsurf: radsurf/radsurf_config.F90:32-113 */
typedef struct ssb200_config {
  int32_t do_sw, do_lw, use_sw_direct_albedo;
  int32_t do_vegetation, do_urban;
  int32_t n_vegetation_region_forest, n_vegetation_region_urban;
  int32_t nsw, nlw; /* = nswinternal, nlwinternal (radsurf_config.F90:260-261) */
  int32_t use_symmetric_vegetation_scale_forest;
  int32_t use_symmetric_vegetation_scale_urban;
  int32_t iverbose;
  double vegetation_isolation_factor_forest;
  double vegetation_isolation_factor_urban;
  double min_vegetation_fraction;
  double min_building_fraction;
  ssb200_legendre_gauss lg_sw_forest, lg_sw_urban, lg_lw_forest, lg_lw_urban;
} ssb200_config;

/* canopy_properties_type: radsurf/radsurf_canopy_properties.F90:53-110
 * (only the members dereferenced under radsurf; temperatures stay upstream) */
typedef struct ssb200_canopy_properties {
  int32_t ncol, ntotlay;
  const int32_t *nlay;             /* (ncol) */
  const int32_t *istartlay;        /* (ncol) 1-based */
  const int32_t *i_representation; /* (ncol) */
  const double *cos_sza;           /* (ncol) */
  const double *dz;                /* (ntotlay) */
  const double *building_fraction, *building_scale;        /* (ntotlay) */
  const double *veg_fraction, *veg_scale, *veg_ext;        /* (ntotlay) */
  const double *veg_fsd, *veg_contact_fraction;            /* (ntotlay) */
} ssb200_canopy_properties;

/* sw_spectral_properties_type: radsurf/radsurf_sw_spectral_properties.F90:24-49 */
typedef struct ssb200_sw_spectral_properties {
  int32_t nspec, pad_;
  const double *air_ext, *air_ssa;  /* (nsw,ntotlay) */
  const double *veg_ssa;            /* (nsw,ntotlay) */
  const double *ground_albedo;      /* (nsw,ncol) */
  const double *roof_albedo, *wall_albedo, *wall_specular_frac; /* (nsw,ntotlay) */
  const double *ground_albedo_dir;  /* (nsw,ncol), may be NULL */
  const double *roof_albedo_dir;    /* (nsw,ntotlay), may be NULL */
} ssb200_sw_spectral_properties;

/* lw_spectral_properties_type: radsurf/radsurf_lw_spectral_properties.F90:24-57 */
typedef struct ssb200_lw_spectral_properties {
  int32_t nspec, pad_;
  const double *air_ext, *air_ssa, *clear_air_planck; /* (nlw,ntotlay) */
  const double *veg_ssa, *veg_planck, *veg_air_planck;/* (nlw,ntotlay) */
  const double *ground_emissivity, *ground_emission;  /* (nlw,ncol) */
  const double *roof_emissivity, *wall_emissivity;    /* (nlw,ntotlay) */
  const double *roof_emission, *wall_emission;        /* (nlw,ntotlay) */
} ssb200_lw_spectral_properties;

/* canopy_flux_type: radsurf/radsurf_canopy_flux.F90:27-91 */
typedef struct ssb200_canopy_flux {
  int32_t nspec, ncol, ntotlay, pad_;
  double *ground_dn, *ground_net, *ground_vertical_diff, *top_dn, *top_net; /* (nspec,ncol) */
  double *ground_dn_dir, *top_dn_dir; /* (nspec,ncol), NULL unless use_direct */
  double *ground_sunlit_frac;         /* (ncol) */
  double *roof_in, *roof_net, *wall_in, *wall_net; /* (nspec,ntotlay) */
  double *roof_in_dir, *wall_in_dir;               /* (nspec,ntotlay) */
  double *roof_sunlit_frac, *wall_sunlit_frac;     /* (ntotlay) */
  double *clear_air_abs;                           /* (nspec,ntotlay) */
  double *veg_abs, *veg_air_abs;                   /* (nspec,ntotlay) */
  double *veg_abs_dir;                             /* (nspec,ntotlay) */
  double *veg_sunlit_frac;                         /* (ntotlay) */
  double *flux_dn_layer_top, *flux_up_layer_top;   /* (nspec,ntotlay) */
  double *flux_dn_layer_base, *flux_up_layer_base; /* (nspec,ntotlay) */
  double *flux_dn_dir_layer_top, *flux_dn_dir_layer_base; /* (nspec,ntotlay) */
} ssb200_canopy_flux;

/* boundary_conds_out_type: radsurf/radsurf_boundary_conds_out.F90:24-39 */
typedef struct ssb200_boundary_conds_out {
  double *sw_albedo, *sw_albedo_dir;     /* (nsw,ncol) */
  double *lw_emissivity, *lw_emission;   /* (nlw,ncol) */
} ssb200_boundary_conds_out;

/* ------------------------------------------------------------------------
 * Entry points of libspartacus_b200.so
 * ------------------------------------------------------------------------ */

/* Library / build identification string. */
const char *ssb200_version(void);

/* sizeof() of the ABI structs in declaration order (legendre_gauss, config,
 * canopy_properties, sw_spectral_properties, lw_spectral_properties,
 * canopy_flux, boundary_conds_out): lets a foreign-language binding verify its
 * mirror of this header at load time. */
int ssb200_abi_sizes(int64_t out[7]);

/* Text of the last error raised on the calling thread ("" if none). */
const char *ssb200_last_error(void);

/* Number of CUDA devices visible (0 => every solve call returns
 * SSB200_ERR_NOGPU; there is no CPU fallback). */
int ssb200_device_count(void);

/* Select the CUDA device used by subsequent calls from this process. */
int ssb200_set_device(int device);

/* Replaces legendre_gauss_type%initialize
 * (radtool/radtool_legendre_gauss.F90:52-100,119-170): host-side constant
 * table, once per configuration. */
int ssb200_legendre_gauss_init(int32_t nstream, ssb200_legendre_gauss *lg);

/* Replaces the body of `radsurf` (radsurf/radsurf_interface.F90:20-317).
 * All array pointers are HOST memory in the reference layout.  Columns
 * istartcol..iendcol (1-based, inclusive; <=0 selects the full range like the
 * absent optional arguments, :86-96) are solved on the GPU and the
 * corresponding slices of bc_out and of the four flux objects are written in
 * place; other columns are untouched.  Flux objects may be NULL when the
 * corresponding do_sw/do_lw is false. */
int ssb200_radsurf(const ssb200_config *config,
                   const ssb200_canopy_properties *canopy_props,
                   const ssb200_sw_spectral_properties *sw_spectral_props,
                   const ssb200_lw_spectral_properties *lw_spectral_props,
                   ssb200_boundary_conds_out *bc_out,
                   int32_t istartcol, int32_t iendcol,
                   ssb200_canopy_flux *sw_norm_dir,
                   ssb200_canopy_flux *sw_norm_diff,
                   ssb200_canopy_flux *lw_internal,
                   ssb200_canopy_flux *lw_norm);

/* What the reference DRIVER does around `radsurf` for every block of columns
 * (driver/spartacus_surface_driver.F90:206-261), as ONE call that keeps the four
 * normalised flux objects on the device:
 *   calc_simple_spectrum_lw      radsurf/radsurf_simple_spectrum.F90:41-66   (emission from temperatures)
 *   radsurf                      radsurf/radsurf_interface.F90:20-317
 *   sw_norm_dir%scale(top_dir); sw_norm_diff%scale(top_dn - top_dir); sw_flux%sum(...)    driver:250-256
 *   lw_norm%scale(top_dn_lw);   lw_flux%sum(lw_internal, lw_norm)                         driver:258-261
 * plus the defaults read_input fills in when the input file lacks a variable
 * (driver/spartacus_surface_read_input.F90:155-166,258-269,311-344,362-365), evaluated on
 * the device for members passed as NULL:
 *   sw%air_ext, lw%air_ext = 1e-5; sw%air_ssa = 0.999; lw%air_ssa = 0; sw%wall_specular_frac = 0;
 *   sw%roof_albedo_dir = sw%roof_albedo;
 *   canopy_props%veg_contact_fraction = min(1, veg_fraction / max(min_vegetation_fraction, 1 - building_fraction));
 *   lw%{ground,roof,wall}_emission, lw%{clear_air,veg,veg_air}_planck from the temperatures below.
 * Only the inputs that carry information and the two summed flux objects cross PCIe
 * (16 instead of 25 input doubles and 2 instead of 4 flux objects per layer).
 * HOST pointers throughout; every array (nspec, ncol) or (ntotlay), reference layout. */
typedef struct ssb200_driver_inputs {
  const double *top_flux_dn_sw;         /* (nsw, ncol) total downwelling SW at canopy top */
  const double *top_flux_dn_direct_sw;  /* (nsw, ncol) its direct part */
  const double *top_flux_dn_lw;         /* (nlw, ncol) */
  const double *ground_temperature;     /* (ncol)    K; used for NULL members of lw_spectral_props */
  const double *roof_temperature, *wall_temperature;                          /* (ntotlay) */
  const double *clear_air_temperature, *veg_temperature, *veg_air_temperature; /* (ntotlay) */
} ssb200_driver_inputs;

/* sw_flux / lw_flux: the summed flux objects (the members that are allocated decide what is
 * computed, like canopy_flux_type%sum); bc_out as in ssb200_radsurf.  Either flux object may
 * be NULL when the corresponding do_sw / do_lw is false. */
int ssb200_radsurf_fluxes(const ssb200_config *config,
                          const ssb200_canopy_properties *canopy_props,
                          const ssb200_sw_spectral_properties *sw_spectral_props,
                          const ssb200_lw_spectral_properties *lw_spectral_props,
                          const ssb200_driver_inputs *driver_inputs,
                          ssb200_boundary_conds_out *bc_out,
                          int32_t istartcol, int32_t iendcol,
                          ssb200_canopy_flux *sw_flux, ssb200_canopy_flux *lw_flux);

/* Single-precision storage variant: what a `-DSINGLE_PRECISION` build of the reference
 * (jprb = real32, utilities/parkind1.F90:45-49; Makefile:41-45) passes.  Same members as the
 * double-precision structs with `float` arrays (the config struct, whose reals are scalars, is
 * shared: the shim widens them).  The arrays cross PCIe as float (half the bytes), are widened on
 * the device, the solve runs in FP64 exactly as ssb200_radsurf does - a superset of the
 * reference's rule that only the eigen-decomposition works in double
 * (radtool/radtool_eigen_decomposition.F90:55-58) - and every output is the FP64 result rounded
 * to nearest float.  HOST pointers; same return convention as ssb200_radsurf. */
typedef struct ssb200_canopy_properties_sp {
  int32_t ncol, ntotlay;
  const int32_t *nlay, *istartlay, *i_representation;
  const float *cos_sza;
  const float *dz;
  const float *building_fraction, *building_scale;
  const float *veg_fraction, *veg_scale, *veg_ext;
  const float *veg_fsd, *veg_contact_fraction;
} ssb200_canopy_properties_sp;
typedef struct ssb200_sw_spectral_properties_sp {
  int32_t nspec, pad_;
  const float *air_ext, *air_ssa;
  const float *veg_ssa;
  const float *ground_albedo;
  const float *roof_albedo, *wall_albedo, *wall_specular_frac;
  const float *ground_albedo_dir;
  const float *roof_albedo_dir;
} ssb200_sw_spectral_properties_sp;
typedef struct ssb200_lw_spectral_properties_sp {
  int32_t nspec, pad_;
  const float *air_ext, *air_ssa, *clear_air_planck;
  const float *veg_ssa, *veg_planck, *veg_air_planck;
  const float *ground_emissivity, *ground_emission;
  const float *roof_emissivity, *wall_emissivity;
  const float *roof_emission, *wall_emission;
} ssb200_lw_spectral_properties_sp;
typedef struct ssb200_canopy_flux_sp {
  int32_t nspec, ncol, ntotlay, pad_;
  float *ground_dn, *ground_net, *ground_vertical_diff, *top_dn, *top_net;
  float *ground_dn_dir, *top_dn_dir;
  float *ground_sunlit_frac;
  float *roof_in, *roof_net, *wall_in, *wall_net;
  float *roof_in_dir, *wall_in_dir;
  float *roof_sunlit_frac, *wall_sunlit_frac;
  float *clear_air_abs;
  float *veg_abs, *veg_air_abs;
  float *veg_abs_dir;
  float *veg_sunlit_frac;
  float *flux_dn_layer_top, *flux_up_layer_top;
  float *flux_dn_layer_base, *flux_up_layer_base;
  float *flux_dn_dir_layer_top, *flux_dn_dir_layer_base;
} ssb200_canopy_flux_sp;
typedef struct ssb200_boundary_conds_out_sp {
  float *sw_albedo, *sw_albedo_dir;
  float *lw_emissivity, *lw_emission;
} ssb200_boundary_conds_out_sp;

int ssb200_radsurf_sp(const ssb200_config *config,
                      const ssb200_canopy_properties_sp *canopy_props,
                      const ssb200_sw_spectral_properties_sp *sw_spectral_props,
                      const ssb200_lw_spectral_properties_sp *lw_spectral_props,
                      ssb200_boundary_conds_out_sp *bc_out,
                      int32_t istartcol, int32_t iendcol,
                      ssb200_canopy_flux_sp *sw_norm_dir,
                      ssb200_canopy_flux_sp *sw_norm_diff,
                      ssb200_canopy_flux_sp *lw_internal,
                      ssb200_canopy_flux_sp *lw_norm);

/* ssb200_radsurf_fluxes for a `-DSINGLE_PRECISION` host: the reference driver's sequence
 * (driver/spartacus_surface_driver.F90:206-261, as ssb200_radsurf_fluxes above) with float arrays.
 * ssb200_driver_inputs_sp has the members of ssb200_driver_inputs as `const float *`.  NULL members
 * take read_input's defaults and the LW emission is derived from the temperatures exactly as in
 * ssb200_radsurf_fluxes.  The arrays cross PCIe as float (half the bytes of the double entry), are
 * widened on the device, the solve, the sigma T^4 emission and the scale + sum run in FP64, and every
 * output is the FP64 result rounded to nearest float: bit-equal to ssb200_radsurf_fluxes on the widened
 * inputs followed by a cast.  HOST pointers; same return convention as ssb200_radsurf. */
typedef struct ssb200_driver_inputs_sp {
  const float *top_flux_dn_sw;
  const float *top_flux_dn_direct_sw;
  const float *top_flux_dn_lw;
  const float *ground_temperature;
  const float *roof_temperature, *wall_temperature;
  const float *clear_air_temperature, *veg_temperature, *veg_air_temperature;
} ssb200_driver_inputs_sp;

int ssb200_radsurf_fluxes_sp(const ssb200_config *config,
                             const ssb200_canopy_properties_sp *canopy_props,
                             const ssb200_sw_spectral_properties_sp *sw_spectral_props,
                             const ssb200_lw_spectral_properties_sp *lw_spectral_props,
                             const ssb200_driver_inputs_sp *driver_inputs,
                             ssb200_boundary_conds_out_sp *bc_out,
                             int32_t istartcol, int32_t iendcol,
                             ssb200_canopy_flux_sp *sw_flux, ssb200_canopy_flux_sp *lw_flux);

/* Device-resident variant.  The three per-column index arrays of
 * `canopy_props` (nlay, istartlay, i_representation) stay HOST pointers (they
 * define the launch plan, which is cached between calls while they do not
 * change); every double array in every struct is a DEVICE pointer in the same
 * reference layout.  Work is enqueued on `stream` (a cudaStream_t passed as
 * void*; NULL = default stream) and the call returns without synchronising;
 * `status_out` (device int32[1], may be NULL) receives the count of flagged
 * problems.  Calls share one context (scratch, plan buffers): a call on a
 * stream other than the previous call's waits (on the device, through an
 * event) for that call's kernels, so results are correct from any stream, but
 * calls do not overlap each other. */
int ssb200_radsurf_device(const ssb200_config *config,
                          const ssb200_canopy_properties *canopy_props,
                          const ssb200_sw_spectral_properties *sw_spectral_props,
                          const ssb200_lw_spectral_properties *lw_spectral_props,
                          ssb200_boundary_conds_out *bc_out,
                          int32_t istartcol, int32_t iendcol,
                          ssb200_canopy_flux *sw_norm_dir,
                          ssb200_canopy_flux *sw_norm_diff,
                          ssb200_canopy_flux *lw_internal,
                          ssb200_canopy_flux *lw_norm,
                          void *stream, int32_t *status_out);

/* ssb200_radsurf_device for float device arrays: replaces the body of `radsurf`
 * (radsurf/radsurf_interface.F90:20-317) for a `-DSINGLE_PRECISION` caller whose arrays live in HBM.
 * Every float array is a DEVICE pointer; nlay, istartlay and i_representation stay HOST arrays.  The
 * call is asynchronous on `stream`, shares the one context of the other entries and is ordered against
 * calls from other streams exactly as ssb200_radsurf_device.  The solve runs in FP64 and every output
 * is the FP64 result rounded to nearest float: bit-equal to ssb200_radsurf_device on the widened inputs
 * followed by a cast; entries the solve leaves untouched keep the caller's value, and columns outside
 * istartcol..iendcol are not written.  No full double copy of the inputs is made when every per-layer
 * read of the call goes through the level-major staging ("stage_layers", the register-resident kernels
 * of 1-4 streams, no "fused_kernels", no SimpleUrban / InfiniteStreet column): the staging widens and
 * rounds the per-layer arrays as it moves them, and only the per-column members are widened into
 * double buffers of the context.  Otherwise the per-layer arrays of the call's packed layers are
 * widened into double buffers too and rounded back.  Same return convention as ssb200_radsurf_device. */
int ssb200_radsurf_device_sp(const ssb200_config *config,
                             const ssb200_canopy_properties_sp *canopy_props,
                             const ssb200_sw_spectral_properties_sp *sw_spectral_props,
                             const ssb200_lw_spectral_properties_sp *lw_spectral_props,
                             ssb200_boundary_conds_out_sp *bc_out,
                             int32_t istartcol, int32_t iendcol,
                             ssb200_canopy_flux_sp *sw_norm_dir,
                             ssb200_canopy_flux_sp *sw_norm_diff,
                             ssb200_canopy_flux_sp *lw_internal,
                             ssb200_canopy_flux_sp *lw_norm,
                             void *stream, int32_t *status_out);

/* ssb200_radsurf_fluxes for a caller whose arrays live in HBM: the reference driver's sequence around
 * radsurf (driver/spartacus_surface_driver.F90:206-261) - calc_simple_spectrum_lw, radsurf, scale of the
 * normalised fluxes by the top-of-canopy fluxes and sum into sw_flux / lw_flux - in one asynchronous call.
 * Same semantics as ssb200_radsurf_fluxes: the members of sw_flux / lw_flux that are allocated decide what
 * is computed, NULL members of the property structs take read_input's defaults, and NULL emission /
 * Planck members are sigma [emissivity] T^4 of the temperatures in `driver_inputs`.  Every array, the
 * members of `driver_inputs` included, is a DEVICE pointer; nlay, istartlay and i_representation stay
 * HOST arrays, as for ssb200_radsurf_device.  The call is enqueued on `stream`, shares the one context of
 * the other entries, is ordered against calls from other streams and fills `status_out` exactly as
 * ssb200_radsurf_device.  Columns outside istartcol..iendcol are not written, and per-layer entries only
 * for the layers of in-range, non-Flat columns; unlike the host entry the packed layers of the selected
 * columns need not be contiguous.  The caller's arrays are never written except the outputs: defaults and
 * emission go to buffers of the context.
 * The four normalised flux objects are never formed in the caller's layout.  When every per-layer write
 * of the call goes through the level-major staging ("stage_layers", the register-resident kernels of 1-4
 * streams, no "fused_kernels", no SimpleUrban / InfiniteStreet column), the staging scatter writes the
 * scaled sum of both objects straight into sw_flux / lw_flux; otherwise the objects are held in buffers
 * of the context for the call's columns and layers and summed after the solve.  Either way the result is
 * bit-equal to ssb200_radsurf_fluxes on the same inputs, and to ssb200_radsurf_device followed by
 * ssb200_canopy_flux_scale_device and ssb200_canopy_flux_sum_device on zeroed normalised objects. */
int ssb200_radsurf_fluxes_device(const ssb200_config *config,
                                 const ssb200_canopy_properties *canopy_props,
                                 const ssb200_sw_spectral_properties *sw_spectral_props,
                                 const ssb200_lw_spectral_properties *lw_spectral_props,
                                 const ssb200_driver_inputs *driver_inputs,
                                 ssb200_boundary_conds_out *bc_out,
                                 int32_t istartcol, int32_t iendcol,
                                 ssb200_canopy_flux *sw_flux, ssb200_canopy_flux *lw_flux,
                                 void *stream, int32_t *status_out);

/* ssb200_radsurf_fluxes_device for float (single-precision) HBM arrays, as a -DSINGLE_PRECISION host
 * model holds them: every real array, the members of `driver_inputs` included, is a float DEVICE pointer;
 * nlay, istartlay and i_representation stay HOST arrays.  Stream, ordering against other streams,
 * `status_out`, the columns and layers written and the return convention are those of
 * ssb200_radsurf_fluxes_device, and non-contiguous packed layers are accepted.
 * The solve, the emission, the defaults of NULL members and the scale + sum run in FP64 on the float
 * inputs widened exactly, and every output is rounded once to nearest float: it equals the output of
 * ssb200_radsurf_fluxes_device on the widened inputs, cast to float, and on contiguous layouts that of
 * ssb200_radsurf_fluxes_sp on the same arrays.  read_input's defaults, sigma T^4 and the default
 * veg_contact_fraction are held as doubles in buffers of the context, never rounded to float.
 * The per-column members, bc_out and the top-of-canopy fluxes are widened into double buffers of the
 * context for the call's columns (bc_out is rounded back).  When every per-layer access of the call goes
 * through the level-major staging (same condition as ssb200_radsurf_fluxes_device), the staging widens the
 * per-layer inputs as it gathers them and its summing scatter rounds into sw_flux / lw_flux; otherwise
 * the per-layer inputs of the call's packed layers are widened into double buffers too. */
int ssb200_radsurf_fluxes_device_sp(const ssb200_config *config,
                                    const ssb200_canopy_properties_sp *canopy_props,
                                    const ssb200_sw_spectral_properties_sp *sw_spectral_props,
                                    const ssb200_lw_spectral_properties_sp *lw_spectral_props,
                                    const ssb200_driver_inputs_sp *driver_inputs,
                                    ssb200_boundary_conds_out_sp *bc_out,
                                    int32_t istartcol, int32_t iendcol,
                                    ssb200_canopy_flux_sp *sw_flux, ssb200_canopy_flux_sp *lw_flux,
                                    void *stream, int32_t *status_out);

/* Number of kernels launched by this process through the library so far
 * (bench.py reports the per-step delta as `gpu_launches`). */
int64_t ssb200_kernel_launch_count(void);

/* Time (ms, CUDA events on the library's launch stream) spent in the most
 * recent ssb200_radsurf_device call, split per kernel family:
 * out[0]=layer-matrix SW, out[1]=sweep SW, out[2]=layer-matrix LW,
 * out[3]=sweep LW, out[4]=other (flat/simple urban/zero fill).  Only filled
 * when profiling was enabled with ssb200_set_profiling(1) (which inserts
 * events and synchronises at the end of the call). */
int ssb200_set_profiling(int enable);
int ssb200_last_kernel_times_ms(double out[5]);
/* Launches per kernel family in that call (same order). */
int ssb200_last_kernel_counts(int64_t out[5]);

/* Tuning knobs (results never depend on them beyond rounding; defaults in brackets):
 *   "scratch_budget_bytes"  device scratch per launch chunk and scratch lane [0 = automatic: a quarter
 *                           of the free memory, at most 12 GiB]
 *   "fast_kernels"          [1] register-resident kernels where a configuration has them (1-4 streams);
 *                           0 = the generic one-thread-per-problem kernels everywhere (TEST-ONLY: they are the
 *                           correctness path of 8 streams, not a tuned one)
 *   "partition_layers"      [1] group layer problems by solved sub-block (needed by the fast layer kernels)
 *   "stage_layers"          [1] level-major staging of the per-layer arrays of a chunk (gather / scatter)
 *   "sort_columns"          [1] process the columns of a launch ordered by their segment pattern inside groups
 *   "sort_group"            [16384] of this many neighbours (0 = the whole chunk)
 *   "concurrent_passes"     [1] shortwave and longwave pass on two streams with separate scratch
 *   "pipeline"              [1] host entries upload, solve and download blocks of columns as three
 *   "pipeline_max_blocks"   [16] overlapping stages (effective with pinned host memory)
 *   "record_sweeps"         [0] measured alternative: operator-record sweeps (1 and 2 streams)
 *   "fused_kernels"         [0] measured alternative: column-resident kernels (1 and 2 streams), with
 *                           "fused_sort", "fused_sort_group", "fused_blocks_per_sm", "fused_sync", "fused_l2_persist" */
int ssb200_set_option(const char *name, int64_t value);

/* Release cached plans, scratch and pinned staging buffers. */
int ssb200_release(void);

/* "Next" row f1: canopy_flux_type%scale / %sum / %check on device
 * (radsurf/radsurf_canopy_flux.F90:212-282,399-460,465-542).  Device
 * pointers; nlay/istartlay are host arrays as above. */
int ssb200_canopy_flux_scale_device(ssb200_canopy_flux *flux, const int32_t *nlay,
                                    const int32_t *istartlay,
                                    const double *factor /* device (nspec,ncol) */,
                                    void *stream);
int ssb200_canopy_flux_sum_device(ssb200_canopy_flux *out, const ssb200_canopy_flux *a,
                                  const ssb200_canopy_flux *b, void *stream);
/* residual[ncol] (device) = ground_net + sum(abs terms) - top_net, per
 * column, summed over spectral intervals (radsurf_canopy_flux.F90:502-540). */
int ssb200_canopy_flux_check_device(const ssb200_canopy_flux *flux,
                                    const ssb200_canopy_properties *canopy_props,
                                    double *residual, void *stream);

/* "Next" row f2: the input stage in front of the path on device -
 * calc_simple_spectrum_lw (radsurf/radsurf_simple_spectrum.F90:41-66) and, with the
 * air / vegetation temperatures NULL, lw_spectral_properties_type%calc_monochromatic_emission
 * (radsurf/radsurf_lw_spectral_properties.F90:161-199): broadband sigma T^4 emission and
 * Planck arrays from temperatures and emissivities (interval 1 of (nspec, .) arrays), so that
 * only the temperatures have to cross PCIe.  Device pointers; a NULL temperature skips the
 * members it feeds.  Columns istartcol..iendcol (1-based, 0 = all) and the packed layers
 * ilay1..ilay2 (1-based, as computed by the reference from istartlay/nlay; ilay2 < ilay1 = none). */
int ssb200_calc_simple_spectrum_lw_device(ssb200_lw_spectral_properties *lw, int32_t ncol, int32_t ntotlay,
                                          int32_t istartcol, int32_t iendcol, int32_t ilay1, int32_t ilay2,
                                          const double *ground_temperature, const double *roof_temperature,
                                          const double *wall_temperature, const double *clear_air_temperature,
                                          const double *veg_temperature, const double *veg_air_temperature,
                                          void *stream);

/* FP64 FMA peak micro-benchmark used as roofline denominator by bench.py:
 * returns measured TFLOP/s (2 flop per DFMA) on the current device, <0 on
 * error. */
double ssb200_measure_fp64_peak_tflops(int iters);

#ifdef __cplusplus
}
#endif
#endif /* SPARTACUS_B200_H */
