// ssb_api.cu - kernels and C-ABI entry points of libspartacus_b200.so
// (include/spartacus_b200.h).  sm_100a only; there is no CPU fallback: every
// solve entry returns SSB200_ERR_NOGPU when no CUDA device is present.
#include <cuda_runtime.h>

#include <cub/cub.cuh>
#include <mutex>

#include "ssb_driver.hpp"
#include "ssb_fast.cuh"
#include "ssb_fast_layer.cuh"
#include "ssb_launch.hpp"

namespace ssb {
cudaError_t g_fast_error = cudaSuccess;
}

namespace {

thread_local std::string g_last_error;
std::mutex g_mutex;
long long g_launches = 0;

int fail(int code, const std::string &msg) {
  g_last_error = msg;
  return code;
}

#define SSB_CUDA(call)                                                                           \
  do {                                                                                           \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess)                                                                       \
      return fail(SSB200_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));          \
  } while (0)

// Flat tiles and single-layer urban models (the generic kernels live in ssb_k_ns*_*.cu)
__global__ void k_surface(ssb::SurfaceArgs s, int nsw_threads, int nlw_threads) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nsw_threads) ssb::surface_column_sw(s, t / s.nsw, t % s.nsw);
  if (t < nlw_threads) ssb::surface_column_lw(s, t / s.nlw, t % s.nlw);
}

// sort keys of the columns of one launch chunk (column_segment_key)
// (columns are ordered inside groups of `group` neighbours only: a warp then still touches
// neighbouring lines of the per-column input and output arrays)
// The key is packed into as few bits as it needs - `lbits` for the segment pattern (one bit per
// layer; night-time columns get the largest value) below the group index - so that the radix sort
// runs 3 passes instead of 8: at 131,072 columns per GPU (8-GPU sharding) the sort is latency, not
// bandwidth.  T: element type of the per-layer fractions (float: ssb200_radsurf_device_sp).
template <class T>
__global__ void k_column_keys(ssb::ClassArgs a, unsigned long long *keys, int group, int lbits) {
  const int ic = blockIdx.x * blockDim.x + threadIdx.x;
  if (ic >= a.ncols) return;
  const unsigned long long all = (1ull << lbits) - 1ull;
  const unsigned pattern = ssb::column_segment_key<T>(a, a.cols[ic]);
  const unsigned long long k = (pattern == 0xffffffffu) ? all : ((unsigned long long)pattern & (all >> 1));
  keys[ic] = ((unsigned long long)(ic / group) << lbits) | k;
}

// ---------------------------------------------------------------------------
// canopy_flux_type%scale / %sum / %check on device (SURVEY §8 row f1)
// ---------------------------------------------------------------------------
struct FieldList {
  double *p[32];
  const double *a[32], *b[32];
  int per_layer[32];  // 1: (nspec, ntotlay), 0: (nspec, ncol)
  int spectral[32];
  int n;
};

__global__ void k_scale(FieldList fl, const double *factor, const int *lay2col, int nspec, long ncol, long ntotlay) {
  const long t = blockIdx.x * (long)blockDim.x + threadIdx.x;
  for (int f = 0; f < fl.n; ++f) {
    const long cnt = (fl.per_layer[f] ? ntotlay : ncol) * nspec;
    if (t < cnt) {
      const long idx = t / nspec;
      const int g = (int)(t % nspec);
      const long col = fl.per_layer[f] ? lay2col[idx] : idx;
      fl.p[f][t] = factor[g + (long)nspec * col] * fl.p[f][t];
    }
  }
}

__global__ void k_sum(FieldList fl, int nspec, long ncol, long ntotlay) {
  const long t = blockIdx.x * (long)blockDim.x + threadIdx.x;
  for (int f = 0; f < fl.n; ++f) {
    const long cnt = (fl.per_layer[f] ? ntotlay : ncol) * (fl.spectral[f] ? nspec : 1);
    if (t < cnt) fl.p[f][t] = fl.a[f][t] + fl.b[f][t];
  }
}

__global__ void k_check(ssb200_canopy_flux f, const int *nlay, const int *istartlay, const int *irep, int ncol,
                        double *residual) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= ncol) return;
  const int ns = f.nspec;
  const int l1 = istartlay[col] - 1, nl = nlay[col], rep = irep[col];
  auto sum_col = [&](const double *p) {
    double s = 0.0;
    for (int g = 0; g < ns; ++g) s += p[g + (size_t)ns * col];
    return s;
  };
  auto sum_lay = [&](const double *p) {
    double s = 0.0;
    if (p)
      for (int l = 0; l < nl; ++l)
        for (int g = 0; g < ns; ++g) s += p[g + (size_t)ns * (l1 + l)];
    return s;
  };
  const double ground_net = sum_col(f.ground_net), top_net = sum_col(f.top_net);
  const double clear = (rep != SSB200_TILE_FLAT) ? sum_lay(f.clear_air_abs) : 0.0;
  double roof = 0.0, wall = 0.0, veg = 0.0, vegair = 0.0;
  if (rep == SSB200_TILE_URBAN || rep == SSB200_TILE_VEGETATED_URBAN || rep == SSB200_TILE_SIMPLE_URBAN ||
      rep == SSB200_TILE_INFINITE_STREET) {
    roof = sum_lay(f.roof_net);
    wall = sum_lay(f.wall_net);
  }
  if (rep == SSB200_TILE_FOREST || rep == SSB200_TILE_VEGETATED_URBAN) {
    veg = sum_lay(f.veg_abs);
    vegair = sum_lay(f.veg_air_abs);
  }
  residual[col] = ground_net + clear + wall + roof + veg + vegair - top_net;
}

// sigma * emissivity * T^4 (emissivity NULL: 1) for elements [i0, i1) of (nspec, .) arrays, interval 1.
// T: element type of the temperatures and emissivities (float inputs are widened exactly; the output and
// the arithmetic stay FP64, so a float caller gets the emission of the double entry on widened inputs).
template <class T>
__global__ void k_sigma_t4(double *out, const T *emissivity, const T *temperature, int nspec, long i0, long i1) {
  const long i = i0 + blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i >= i1) return;
  const double t = (double)temperature[i], t2 = t * t;
  const double sb = 5.67037321e-8;  // radtool/radiation_constants.F90:26
  out[(size_t)nspec * i] = emissivity ? (sb * (double)emissivity[(size_t)nspec * i]) * (t2 * t2) : sb * (t2 * t2);
}

// ---- single-precision storage variant: float <-> double on the device (ssb200_radsurf_sp) ----
__global__ void k_f2d(double *dst, const float *src, size_t n) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (double)src[i];
}
__global__ void k_d2f(float *dst, const double *src, size_t n) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) dst[i] = (float)src[i];  // round to nearest even
}

// ---- ssb200_radsurf_device_sp: float device arrays around the FP64 solve ----------------------
// element ranges [lo, hi) of a list of arrays, widened (d = f, exact) before the solve or rounded to
// nearest (f = d) after it, one launch per direction
constexpr int kConvMax = 48;
struct ConvList {
  float *f[kConvMax];
  double *d[kConvMax];
  long lo[kConvMax], hi[kConvMax];
  int n;
};
struct ConvArray {
  float *f;
  double *d;
  long lo, hi;
  bool out;  // rounded back after the solve
};
template <bool ROUND>
__global__ void k_convert(ConvList cl) {
  const long t = blockIdx.x * (long)blockDim.x + threadIdx.x;
  for (int k = 0; k < cl.n; ++k) {
    const long i = cl.lo[k] + t;
    if (i >= cl.hi[k]) continue;
    if (ROUND)
      cl.f[k][i] = __double2float_rn(cl.d[k][i]);
    else
      cl.d[k][i] = (double)cl.f[k][i];
  }
}

// ---- stages around radsurf for ssb200_radsurf_fluxes ----------------------------------------
__global__ void k_fill(double *p, double v, long i0, long i1) {
  const long i = i0 + blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i < i1) p[i] = v;
}
// read_input's default veg_contact_fraction (driver/spartacus_surface_read_input.F90:155-166); T: element
// type of the fractions (float: widened exactly, the result stays FP64)
template <class T>
__global__ void k_vcf_default(double *vcf, const T *vf, const T *bf, double min_veg, long i0, long i1) {
  const long i = i0 + blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i < i1) vcf[i] = fmin(1.0, (double)vf[i] / fmax(min_veg, 1.0 - (double)bf[i]));
}
__global__ void k_lay2col(const int *nlay, const int *istartlay, const int *irep, int ncol, int *lay2col) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= ncol || irep[j] == SSB200_TILE_FLAT) return;
  const int l0 = istartlay[j] - 1;
  for (int l = 0; l < nlay[j]; ++l) lay2col[l0 + l] = j;
}
// out = a * fa + b * fb per (interval, column) factor, every product and the sum rounded separately
// so that the result equals canopy_flux_type%scale followed by %sum bit for bit
// (radsurf/radsurf_canopy_flux.F90:212-282,399-460).  fa NULL: 1.  fb_minus non-NULL: fb - fb_minus.
// Non-spectral members (sunlit fractions) are summed unscaled.  Window: columns [c0, c1), layers [l0, l1);
// a layer of the window is skipped unless a column of [c0, c1) owns it (lay2col: -1 for the layers of no
// non-Flat column), so packed layouts whose layers are not contiguous leave other columns' layers alone.
// R: element type of the summed object (float: ssb200_radsurf_fluxes_device_sp; the FP64 result is rounded
// once to nearest).
__device__ __forceinline__ void store_rounded(double *p, double v) { *p = v; }
__device__ __forceinline__ void store_rounded(float *p, double v) { *p = __double2float_rn(v); }
template <class R>
__global__ void k_scale_sum(FieldList fl, const double *fa, const double *fb, const double *fb_minus,
                            const int *lay2col, int nspec, long c0, long c1, long l0, long l1) {
  const long t = blockIdx.x * (long)blockDim.x + threadIdx.x;
  for (int f = 0; f < fl.n; ++f) {
    const int w = fl.spectral[f] ? nspec : 1;
    const long lo = (fl.per_layer[f] ? l0 : c0) * w, hi = (fl.per_layer[f] ? l1 : c1) * w;
    const long i = lo + t;
    if (i >= hi) continue;
    const long idx = i / w;
    const long col = fl.per_layer[f] ? lay2col[idx] : idx;
    if (col < c0 || col >= c1) continue;
    const double a = fl.a[f][i], b = fl.b[f][i];
    R *p = reinterpret_cast<R *>(fl.p[f]) + i;
    if (!fl.spectral[f]) {
      store_rounded(p, __dadd_rn(a, b));
      continue;
    }
    const int g = (int)(i % nspec);
    const size_t k = (size_t)g + (size_t)nspec * (size_t)col;
    const double xa = fa ? __dmul_rn(fa[k], a) : a;
    const double fbk = fb_minus ? __dadd_rn(fb[k], -fb_minus[k]) : fb[k];
    store_rounded(p, __dadd_rn(xa, __dmul_rn(fbk, b)));
  }
}

// register-resident independent DFMA chains: FP64 roofline denominator
__global__ void k_fp64_peak(double *out, int iters) {
  double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6,
         a7 = a0 + 7;
  const double m = 1.0000001, c = 1e-7;
  for (int i = 0; i < iters; ++i) {
    a0 = fma(a0, m, c);
    a1 = fma(a1, m, c);
    a2 = fma(a2, m, c);
    a3 = fma(a3, m, c);
    a4 = fma(a4, m, c);
    a5 = fma(a5, m, c);
    a6 = fma(a6, m, c);
    a7 = fma(a7, m, c);
  }
  out[blockIdx.x * (size_t)blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

// ---------------------------------------------------------------------------
// Context: cached device buffers, plan, scratch
// ---------------------------------------------------------------------------
struct DevBuf {
  void *p = nullptr;
  size_t bytes = 0;
  cudaError_t reserve(size_t need) {
    if (need <= bytes) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
    cudaError_t e = cudaMalloc(&p, need);
    if (e == cudaSuccess) bytes = need;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    bytes = 0;
  }
};

// Grow-only pool over one of the context's buffer vectors: the i-th request of a call reuses the i-th
// buffer.  The first allocation error is kept in `rc` (message prefixed by `what`); later requests
// return NULL.
struct Pool {
  std::vector<DevBuf> &bufs;
  const char *what;
  size_t next = 0;
  int rc = 0;
  template <class T>
  T *get(size_t n) {
    if (rc) return nullptr;
    if (next >= bufs.size()) bufs.resize(next + 16);
    const cudaError_t e = bufs[next++].reserve(std::max(n, (size_t)1) * sizeof(T));
    if (e != cudaSuccess) {
      rc = fail(SSB200_ERR_CUDA, std::string(what) + cudaGetErrorString(e));
      return nullptr;
    }
    return (T *)bufs[next - 1].p;
  }
};

struct Context {
  ssb::Plan plan;
  bool plan_uploaded = false;
  long uploaded_generation = -1;
  DevBuf d_nlay, d_istart, d_irep, d_cols, d_status, d_lay2col;
  static constexpr int kLanes = 3;  // host entry: upload / kernel / download streams; scratch: lane 0 device entry, lane 1 host entry
  DevBuf d_scratch[kLanes], d_perm[kLanes], d_sort[kLanes];
  cudaStream_t lane_stream[kLanes] = {nullptr, nullptr, nullptr};
  std::vector<cudaEvent_t> blk_events;  // per pipeline block: upload done, kernels done
  int pipeline = 1;
  int pipeline_max_blocks = 16;
  std::vector<DevBuf> stage;  // staging mirrors of host arrays for ssb200_radsurf
  std::vector<DevBuf> wide;   // double copies of float device arrays for ssb200_radsurf_device_sp
  std::vector<DevBuf> drv;    // defaulted inputs and normalised flux members of ssb200_radsurf_fluxes_device
  cudaStream_t stream = nullptr;
  cudaStream_t own_stream = nullptr;
  size_t budget_doubles = 0;
  bool profiling = false;
  double times_ms[5] = {0, 0, 0, 0, 0};
  long long counts[5] = {0, 0, 0, 0, 0};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t ev_done = nullptr;  // end of the last device-entry call (cross-stream ordering)
  cudaStream_t last_stream = nullptr;
  bool last_stream_valid = false;
  cudaError_t first_error = cudaSuccess;
  int fast_mode = 1;
  size_t l2_set_aside = 0;
  long lay2col_generation = -1;
  // order the columns of a launch by their segment pattern (fast kernels): warps then take one code
  // path per layer, the segment kernels write and the sweeps skip whole 32-byte sectors.  Measured on
  // B200 (1 M columns, S2) TOGETHER with the level-major staging below, which makes the column order
  // irrelevant for the per-layer inputs and outputs: 59.8 -> 50.9 ms per step (without the staging the
  // ordering made the sweeps slower: round 1).
  int sort_columns = 1;
  int sort_group = 16384;  // ... inside groups of this many neighbouring columns (0: the whole chunk); measured 1024 .. 65536: 48.0 / 47.3 (4096) / 47.2 / 46.9 (16384) / 47.0 / 47.2 ms per step
  int partition = 1;  // group layer problems by solved sub-block before the fast layer kernels
  // column-resident kernels (ssb_fused.cuh) where they exist (1 and 2 streams); 0: split path
  // sweeps of the register-resident path at 1 and 2 streams: 0 = interface-state sweeps
  // (ssb_fast_sweeps.cuh), 1 = record sweeps (ssb_fused.cuh MODE 1 / 2)
  // shortwave and longwave pass of a call on two streams (separate scratch; no effect while profiling)
  int concurrent_passes = 1;
  cudaStream_t aux_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int sweep_mode = 0;  // measured on B200 (DESIGN.md): the record sweeps move fewer bytes and are 6 % slower
  // level-major staging of the per-layer arrays of a chunk (ssb_stage.cuh)
  int stage_layers = 1;
  int fused_mode = 0;  // measured on B200 (DESIGN.md section 4.5): 40 % fewer DRAM bytes, 28 % slower - off by default
  int fused_sort = 1;
  int fused_sort_group = 0;   // 0: the whole chunk
  int fused_sync = 0;         // block-aligned phases (ssb_fused.cuh: phase_sync): measured, no gain
  int fused_blocks_per_sm = 2;
  int fused_l2_persist = 0;   // pin the private tiles in L2 (access policy window): measured, 25 % slower
  int sm_count = 0;
};
Context g_ctx;

struct CudaBackend {
  Context &cx;
  int lane;
  int pass_lane;            // scratch / perm / sort buffers of the pass being dispatched
  cudaStream_t main_stream; // the stream of the call; the longwave pass may run on cx.aux_stream
  bool forked = false;
  size_t budget;
  bool layer_was_fast = false;  // the chunk's layer kernels were the register-resident ones
  bool f32_layers = false;      // per-layer members are the caller's float arrays (single-precision device entries)
  explicit CudaBackend(Context &c, int lane_ = 0, size_t budget_ = 0)
      : cx(c), lane(lane_), pass_lane(lane_), main_stream(c.stream), budget(budget_ ? budget_ : c.budget_doubles) {}
  // Shortwave pass on the stream of the call, longwave pass on an auxiliary stream with its own
  // scratch (lane 2): the tails of one pass's launches are filled by the other's blocks, and the
  // memory-bound sweeps of one overlap the FP64-bound layer kernels of the other.
  void fork_passes() {
    if (!cx.concurrent_passes || cx.profiling || cx.first_error != cudaSuccess) return;
    if (!cx.aux_stream && cudaStreamCreateWithFlags(&cx.aux_stream, cudaStreamNonBlocking) != cudaSuccess) return;
    if (!cx.ev_fork) {
      if (cudaEventCreateWithFlags(&cx.ev_fork, cudaEventDisableTiming) != cudaSuccess) return;
      if (cudaEventCreateWithFlags(&cx.ev_join, cudaEventDisableTiming) != cudaSuccess) return;
    }
    cudaEventRecord(cx.ev_fork, main_stream);
    cudaStreamWaitEvent(cx.aux_stream, cx.ev_fork, 0);
    forked = true;
  }
  void begin_pass(bool lw) {
    if (!forked) return;
    cx.stream = lw ? cx.aux_stream : main_stream;
    pass_lane = lw ? 2 : lane;
  }
  void end_passes() {
    if (forked) {
      cudaEventRecord(cx.ev_join, cx.aux_stream);
      cudaStreamWaitEvent(main_stream, cx.ev_join, 0);
      forked = false;
    }
    cx.stream = main_stream;
    pass_lane = lane;
  }
  const int *dev_cols(const ssb::Plan &, size_t off) { return (const int *)cx.d_cols.p + off; }
  // columns of the chunk ordered by their segment pattern (device radix sort, stable)
  // (always for the column-resident kernels: a thread walks the layers of its column, so the
  // warps only stay on one code path when neighbouring columns have the same segment pattern)
  const int *order_chunk(const ssb::ClassArgs &a, const int *) {
    const bool want = a.fused ? cx.fused_sort != 0 : (cx.sort_columns && cx.partition);
    if (!cx.fast_mode || !want || a.ncols < 64 || a.cfg.ns > 4 || cx.first_error != cudaSuccess)
      return a.cols;
    const size_t n = (size_t)a.ncols, pad = (n + 63) & ~(size_t)63;
    typedef unsigned long long Key;
    size_t temp_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, (const Key *)nullptr, (Key *)nullptr, (const int *)nullptr,
                                    (int *)nullptr, (int)n, 0, 64, cx.stream);
    temp_bytes = (temp_bytes + 255) & ~(size_t)255;
    if (cx.d_sort[pass_lane].reserve(temp_bytes + pad * (2 * sizeof(Key) + sizeof(int))) != cudaSuccess) {
      cudaGetLastError();
      return a.cols;
    }
    char *base = (char *)cx.d_sort[pass_lane].p;
    Key *keys = (Key *)(base + temp_bytes), *keys_out = keys + pad;
    int *cols_out = (int *)(keys_out + pad);
    const int group = a.fused ? (cx.fused_sort_group > 0 ? cx.fused_sort_group : 0x7fffffff)
                              : (cx.sort_group > 0 ? cx.sort_group : 0x7fffffff);
    const int lbits = (a.lmax < 31 ? a.lmax : 31) + 1;
    int gbits = 0;
    for (size_t ngroups = (n + (size_t)group - 1) / (size_t)group; ((size_t)1 << gbits) < ngroups; ++gbits) {
    }
    // (the key reads building_fraction and veg_fraction only, which the driver-sequence entries never
    // replace by a double default: with float layers they are always the caller's float arrays)
    if (f32_layers)
      k_column_keys<float><<<(unsigned)((n + 127) / 128), 128, 0, cx.stream>>>(a, keys, group, lbits);
    else
      k_column_keys<double><<<(unsigned)((n + 127) / 128), 128, 0, cx.stream>>>(a, keys, group, lbits);
    cub::DeviceRadixSort::SortPairs(base, temp_bytes, keys, keys_out, a.cols, cols_out, (int)n, 0, lbits + gbits,
                                    cx.stream);
    g_launches += 2;
    check_launch();
    return cols_out;
  }
  const int *dev_nlay() { return (const int *)cx.d_nlay.p; }
  const int *dev_istartlay() { return (const int *)cx.d_istart.p; }
  const int *dev_irep() { return (const int *)cx.d_irep.p; }
  int *dev_status() { return (int *)cx.d_status.p; }
  size_t scratch_budget_doubles() { return budget; }
  double *scratch(size_t n) {
    cudaError_t e = cx.d_scratch[pass_lane].reserve(n * sizeof(double));
    if (e != cudaSuccess && cx.first_error == cudaSuccess) cx.first_error = e;
    return (double *)cx.d_scratch[pass_lane].p;
  }
  void tick(int family, bool start) {
    if (!cx.profiling) return;
    if (start) {
      cudaEventRecord(cx.ev0, cx.stream);
    } else {
      cudaEventRecord(cx.ev1, cx.stream);
      cudaEventSynchronize(cx.ev1);
      float ms = 0;
      cudaEventElapsedTime(&ms, cx.ev0, cx.ev1);
      cx.times_ms[family] += ms;
      cx.counts[family] += 1;
    }
  }
  void check_launch() {
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = ssb::g_fast_error;
    ssb::g_fast_error = cudaSuccess;
    if (e != cudaSuccess && cx.first_error == cudaSuccess) cx.first_error = e;
  }
  template <class F>
  void launch(F launcher, const ssb::ClassArgs &a, long nt, int family) {
    if (nt <= 0 || cx.first_error != cudaSuccess) return;
    tick(family, true);
    launcher(a, nt, cx.stream);
    check_launch();
    tick(family, false);
  }
  template <int NS>
  void layer_sw(const ssb::ClassArgs &a, long nt) {
    if (cx.fast_mode && nt > 0 && cx.first_error == cudaSuccess) {
      tick(0, true);
      ssb::ClassArgs b = a;
      if (cx.partition && cx.d_perm[pass_lane].reserve(sizeof(int) * (3 * (size_t)nt + 4)) == cudaSuccess) {
        b.perm_count = (int *)cx.d_perm[pass_lane].p;
        b.perm = b.perm_count + 4;
      }
      const bool done = ssb::fast_layer_sw<NS>(b, nt, cx.stream);
      layer_was_fast = done;
      if (done && b.perm) g_launches += 3;
      if (done) check_launch();
      tick(0, false);
      if (done) return;
    }
    if (a.lstride) {  // staged arrays are only understood by the register-resident kernels
      if (cx.first_error == cudaSuccess) cx.first_error = cudaErrorNotSupported;
      return;
    }
    launch(ssb::launch_layer_sw<NS>, a, nt, 0);
  }
  template <int NS>
  void layer_lw(const ssb::ClassArgs &a, long nt) {
    if (cx.fast_mode && nt > 0 && cx.first_error == cudaSuccess) {
      tick(2, true);
      ssb::ClassArgs b = a;
      if (cx.partition && cx.d_perm[pass_lane].reserve(sizeof(int) * (3 * (size_t)nt + 4)) == cudaSuccess) {
        b.perm_count = (int *)cx.d_perm[pass_lane].p;
        b.perm = b.perm_count + 4;
      }
      const bool done = ssb::fast_layer_lw<NS>(b, nt, cx.stream);
      layer_was_fast = done;
      if (done && b.perm) g_launches += 3;
      if (done) check_launch();
      tick(2, false);
      if (done) return;
    }
    if (a.lstride) {
      if (cx.first_error == cudaSuccess) cx.first_error = cudaErrorNotSupported;
      return;
    }
    launch(ssb::launch_layer_lw<NS>, a, nt, 2);
  }
  // The planner sizes the interface scratch of a staged chunk by the register-resident state alone
  // (run_class); the generic sweeps need their larger one and must never run on a smaller area.
  static bool generic_sweep_scratch(const ssb::ClassArgs &a, bool lw) {
    const ssb::SolveCfg &c = a.cfg;
    const int n = c.nreg * c.ns, d = c.nreg, nrb = c.urban ? c.nreg + 1 : c.nreg, m = nrb * c.ns;
    return a.ne_sweep >= (lw ? ssb::lw_sweep_elems(n, m, c.nreg, nrb) : ssb::sw_sweep_elems(n, d, m, nrb, c.nreg, nrb));
  }
  template <int NS>
  void sweeps_sw(const ssb::ClassArgs &a, long nt) {
    // the register-resident sweeps read what the partition pass of the layer kernels prepared
    if (cx.fast_mode && (layer_was_fast || a.lmax == 0) && nt > 0 && cx.first_error == cudaSuccess) {
      tick(1, true);
      const bool done = ssb::fast_sweeps_sw<NS>(a, nt, cx.stream);
      if (done) check_launch();
      tick(1, false);
      if (done) return;
    }
    if (a.lstride || !generic_sweep_scratch(a, false)) {
      if (cx.first_error == cudaSuccess) cx.first_error = cudaErrorNotSupported;
      return;
    }
    launch(ssb::launch_sweeps_sw<NS>, a, nt, 1);
  }
  template <int NS>
  void sweeps_lw(const ssb::ClassArgs &a, long nt) {
    if (cx.fast_mode && (layer_was_fast || a.lmax == 0) && nt > 0 && cx.first_error == cudaSuccess) {
      tick(3, true);
      const bool done = ssb::fast_sweeps_lw<NS>(a, nt, cx.stream);
      if (done) check_launch();
      tick(3, false);
      if (done) return;
    }
    if (a.lstride || !generic_sweep_scratch(a, true)) {
      if (cx.first_error == cudaSuccess) cx.first_error = cudaErrorNotSupported;
      return;
    }
    launch(ssb::launch_sweeps_lw<NS>, a, nt, 3);
  }
  bool fused_shape(const ssb::SolveCfg &c, bool lw, int *pe, int *oe, int *geo) {
    if (!cx.fast_mode || !cx.fused_mode || c.ns > 2) return false;
    return ssb::fused_shape(c, lw, pe, oe, geo);
  }
  bool stage_supported(const ssb::SolveCfg &c) {
    return cx.fast_mode && cx.partition && cx.stage_layers && c.ns <= 4 && c.nspec <= 1024;
  }
  void stage(const ssb::StageArgs &s, bool scatter, bool lw) {
    if (cx.first_error != cudaSuccess) return;
    const int fam = 4;  // booked with the surface kernels ("surface" family of ssb200_last_kernel_times_ms)
    (void)lw;
    tick(fam, true);
    long n = 0;
    ssb::stage_launch(s, scatter, cx.stream, &n);
    g_launches += n;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess && cx.first_error == cudaSuccess) cx.first_error = e;
    tick(fam, false);
  }
  bool records_shape(const ssb::SolveCfg &c, bool lw, int *oe) {
    if (!cx.fast_mode || cx.sweep_mode != 1 || !cx.partition || c.ns > 2) return false;
    int pe = 0, geo = 0;
    return ssb::fused_shape(c, lw, &pe, oe, &geo);
  }
  void records_run(const ssb::ClassArgs &a, bool lw, long width) {
    if (width <= 0 || cx.first_error != cudaSuccess) return;
    if (!layer_was_fast && a.lmax > 0) {  // the records are built from the register-resident layer scratch
      cx.first_error = cudaErrorNotSupported;
      return;
    }
    const int fam = lw ? 3 : 1;
    tick(fam, true);
    ssb::records_launch(a, lw, width, cx.stream);
    g_launches += 1;  // (check_launch counts one)
    check_launch();
    tick(fam, false);
  }
  int fused_slots() {
    if (cx.sm_count <= 0) {
      int dev = 0, n = 0;
      cudaGetDevice(&dev);
      cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
      cx.sm_count = n > 0 ? n : 148;
    }
    return cx.fused_blocks_per_sm * cx.sm_count;  // __launch_bounds__(128, 2)
  }
  int fused_flags() { return 1 | (cx.fused_sync ? 2 : 0); }
  // The private tiles are re-read and re-written for every layer of every column while the operator
  // records, inputs and outputs stream through L2 once: keep the former resident with a persisting
  // access-policy window on the launch stream (the set-aside is capped by the device limit).
  void l2_window(const void *base, size_t bytes) {
    if (!cx.fused_l2_persist) return;
    int dev = 0, max_persist = 0, max_window = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev);
    cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, dev);
    if (max_persist <= 0 || max_window <= 0) return;
    const size_t set_aside = bytes < (size_t)max_persist ? bytes : (size_t)max_persist;
    if (bytes > 0 && cx.l2_set_aside != set_aside) {
      if (cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, set_aside) == cudaSuccess) cx.l2_set_aside = set_aside;
      cudaGetLastError();
    }
    cudaStreamAttrValue v;
    memset(&v, 0, sizeof(v));
    v.accessPolicyWindow.base_ptr = const_cast<void *>(base);
    v.accessPolicyWindow.num_bytes = bytes < (size_t)max_window ? bytes : (size_t)max_window;
    v.accessPolicyWindow.hitRatio = bytes > 0 ? (float)((double)set_aside / (double)bytes) : 0.0f;
    if (v.accessPolicyWindow.hitRatio > 1.0f) v.accessPolicyWindow.hitRatio = 1.0f;
    v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    v.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
    cudaStreamSetAttribute(cx.stream, cudaStreamAttributeAccessPolicyWindow, &v);
    cudaGetLastError();
  }
  void fused_run(const ssb::ClassArgs &a, bool lw, long width) {
    if (width <= 0 || cx.first_error != cudaSuccess) return;
    const int fam = lw ? 2 : 0;  // booked under the layer families (kernel_times: sw_layer / lw_layer)
    tick(fam, true);
    const long tiles = (width + ssb::kScratchTile - 1) / ssb::kScratchTile;
    const int grid = (int)(tiles < (long)fused_slots() ? tiles : (long)fused_slots());
    l2_window(a.layer, (size_t)grid * (size_t)a.ne_layer * ssb::kScratchTile * sizeof(double));
    ssb::fused_launch(a, lw, width, grid, cx.stream);
    check_launch();
    l2_window(nullptr, 0);
    tick(fam, false);
  }
  void surface(const ssb::SurfaceArgs &s, int nsw_threads, int nlw_threads) {
    const int nt = nsw_threads > nlw_threads ? nsw_threads : nlw_threads;
    if (nt <= 0 || cx.first_error != cudaSuccess) return;
    tick(4, true);
    k_surface<<<(nt + 127) / 128, 128, 0, cx.stream>>>(s, nsw_threads, nlw_threads);
    check_launch();
    tick(4, false);
  }
};

int ensure_device() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return fail(SSB200_ERR_NOGPU, "no CUDA device visible: libspartacus_b200 has no CPU fallback");
  }
  return 0;
}

int upload_plan(Context &cx, const ssb200_canopy_properties &cp) {
  const size_t ncol = (size_t)cp.ncol;
  SSB_CUDA(cx.d_nlay.reserve(sizeof(int) * (ncol + 1)));
  SSB_CUDA(cx.d_istart.reserve(sizeof(int) * (ncol + 1)));
  SSB_CUDA(cx.d_irep.reserve(sizeof(int) * (ncol + 1)));
  SSB_CUDA(cx.d_cols.reserve(sizeof(int) * (cx.plan.all_cols.size() + 1)));
  SSB_CUDA(cudaMemcpyAsync(cx.d_nlay.p, cx.plan.nlay.data(), sizeof(int) * ncol, cudaMemcpyHostToDevice, cx.stream));
  SSB_CUDA(cudaMemcpyAsync(cx.d_istart.p, cx.plan.istartlay.data(), sizeof(int) * ncol, cudaMemcpyHostToDevice,
                           cx.stream));
  SSB_CUDA(cudaMemcpyAsync(cx.d_irep.p, cx.plan.irep.data(), sizeof(int) * ncol, cudaMemcpyHostToDevice, cx.stream));
  SSB_CUDA(cudaMemcpyAsync(cx.d_cols.p, cx.plan.all_cols.data(), sizeof(int) * cx.plan.all_cols.size(),
                           cudaMemcpyHostToDevice, cx.stream));
  // the host vectors must stay unchanged until the copies are done
  SSB_CUDA(cudaStreamSynchronize(cx.stream));
  cx.plan_uploaded = true;
  cx.uploaded_generation = cx.plan.generation;
  return 0;
}

typedef ssb::Dispatcher<CudaBackend>::PassSum PassSum;

// Runs the prepared plan on cx.stream.  prec.f32: the per-layer members of `ca` are float arrays that
// only the level-major staging touches (single-precision device entries, staged route), apart from the
// double buffers in prec.f64.  sum_sw / sum_lw: summing scatter of each pass (ssb200_radsurf_fluxes_device
// and _sp, staged route).
int dispatch_call(Context &cx, const ssb::CallArgs &ca, const ssb::StagePrecision &prec = ssb::StagePrecision(),
                  const PassSum &sum_sw = PassSum(), const PassSum &sum_lw = PassSum()) {
  std::string err;
  CudaBackend be(cx);
  be.f32_layers = prec.f32;
  ssb::Dispatcher<CudaBackend> disp(be);
  disp.precision = prec;
  disp.sum_sw = sum_sw;
  disp.sum_lw = sum_lw;
  const int rc = disp.run(ca, cx.plan, err);
  if (rc) return fail(rc, err);
  if (cx.first_error != cudaSuccess)
    return fail(SSB200_ERR_CUDA, std::string("kernel launch / scratch allocation: ") + cudaGetErrorString(cx.first_error));
  return 0;
}

// End of a device-entry call: status word to the caller, and the event that a later call on another
// stream waits for before it reuses the context's buffers.
int finish_device_call(Context &cx, cudaStream_t stream, int32_t *status_out) {
  if (status_out)
    SSB_CUDA(cudaMemcpyAsync(status_out, cx.d_status.p, sizeof(int), cudaMemcpyDeviceToDevice, stream));
  if (!cx.ev_done) SSB_CUDA(cudaEventCreateWithFlags(&cx.ev_done, cudaEventDisableTiming));
  SSB_CUDA(cudaEventRecord(cx.ev_done, stream));
  cx.last_stream = stream;
  cx.last_stream_valid = true;
  return 0;
}

// Synchronises `s` on scope exit unless disarmed: an error return of a device entry after its first
// launch must not leave work queued on the context's buffers (a later call on another stream, or
// ssb200_release, would not wait for it).
struct Drain {
  cudaStream_t s;
  bool armed = true;
  ~Drain() {
    if (armed) cudaStreamSynchronize(s);
  }
};

// Core of both entry points; all double arrays are device pointers here.
// `blocks`: when non-null the call only prepares (plan, status, budget) and returns the
// clamped 1-based column range in blocks[0..1]; the caller then dispatches column
// windows itself with run_window().
int radsurf_device_locked(Context &cx, const ssb::CallArgs &ca, int istartcol, int iendcol, cudaStream_t stream,
                          int32_t *status_out, int *blocks = nullptr) {
  std::string err;
  int rc = ssb::validate_call(ca, err);
  if (rc) return fail(rc, err);
  const ssb200_canopy_properties &cp = *ca.cp;
  int c1 = istartcol > 0 ? istartcol : 1;
  int c2 = iendcol > 0 ? iendcol : cp.ncol;
  if (c2 > cp.ncol) c2 = cp.ncol;
  if (c1 > c2) return 0;
  cx.stream = stream;
  cx.first_error = cudaSuccess;
  rc = ssb::build_plan(*ca.config, cp, c1 - 1, c2 - 1, cx.plan, err);
  if (rc) {
    cx.plan.valid = false;
    return fail(rc, err);
  }
  rc = ssb::validate_members(ca, cx.plan, err);
  if (rc) return fail(rc, err);
  // One Context (scratch, status word, plan buffers) serves every call: work of an earlier call
  // that is still in flight on ANOTHER stream must finish before this call reuses them.
  if (cx.ev_done && cx.last_stream_valid && cx.last_stream != stream) SSB_CUDA(cudaStreamWaitEvent(stream, cx.ev_done, 0));
  if (cx.plan.generation != cx.uploaded_generation) cx.plan_uploaded = false;
  if (!cx.plan_uploaded) {
    rc = upload_plan(cx, cp);
    if (rc) return rc;
  }
  SSB_CUDA(cx.d_status.reserve(sizeof(int)));
  SSB_CUDA(cudaMemsetAsync(cx.d_status.p, 0, sizeof(int), stream));
  if (cx.budget_doubles == 0) {
    size_t free_b = 0, total_b = 0;
    SSB_CUDA(cudaMemGetInfo(&free_b, &total_b));
    // per scratch lane (two lanes are live when the SW and LW passes run concurrently)
    size_t b = (free_b + cx.d_scratch[0].bytes + cx.d_scratch[1].bytes + cx.d_scratch[2].bytes) / 4;
    const size_t cap = (size_t)12 << 30;  // (more, smaller chunks overlap the two passes better: 47.0 -> 46.7 ms against 24 GiB)
    if (b > cap) b = cap;
    cx.budget_doubles = b / sizeof(double);
  }
  if (cx.profiling) {
    if (!cx.ev0) {
      cudaEventCreate(&cx.ev0);
      cudaEventCreate(&cx.ev1);
    }
    for (double &t : cx.times_ms) t = 0.0;
    for (long long &n : cx.counts) n = 0;
  }
  if (blocks) {
    blocks[0] = c1;
    blocks[1] = c2;
    return 0;
  }
  rc = dispatch_call(cx, ca);
  if (rc) return rc;
  return finish_device_call(cx, stream, status_out);
}

// dispatch the columns [col_lo, col_hi) (0-based) of the prepared plan on one lane
int run_window(Context &cx, const ssb::CallArgs &ca, int lane, size_t budget, int col_lo, int col_hi) {
  std::string err;
  cx.stream = cx.lane_stream[lane];
  CudaBackend be(cx, lane, budget);
  ssb::Dispatcher<CudaBackend> disp(be);
  disp.col_lo = col_lo;
  disp.col_hi = col_hi;
  const int rc = disp.run(ca, cx.plan, err);
  if (rc) return fail(rc, err);
  if (cx.first_error != cudaSuccess)
    return fail(SSB200_ERR_CUDA, std::string("kernel launch / scratch allocation: ") + cudaGetErrorString(cx.first_error));
  return 0;
}

// owner column of every packed layer of the uploaded plan (-1: no non-Flat column owns it), on `st`
int ensure_lay2col(Context &cx, size_t ncol, size_t ntot, cudaStream_t st) {
  if (cx.lay2col_generation == cx.plan.generation) return 0;
  SSB_CUDA(cx.d_lay2col.reserve(sizeof(int) * (ntot + 1)));
  SSB_CUDA(cudaMemsetAsync(cx.d_lay2col.p, 0xff, sizeof(int) * ntot, st));
  if (ncol > 0) {
    k_lay2col<<<(unsigned)((ncol + 127) / 128), 128, 0, st>>>((const int *)cx.d_nlay.p, (const int *)cx.d_istart.p,
                                                               (const int *)cx.d_irep.p, (int)ncol, (int *)cx.d_lay2col.p);
    ++g_launches;
    SSB_CUDA(cudaGetLastError());
  }
  cx.lay2col_generation = cx.plan.generation;
  return 0;
}

// The members of `o` that k_scale / k_sum / k_scale_sum visit.  with_sunlit: also the non-spectral
// members (sunlit fractions); with_layers: also the per-layer ones.  Given `a`, a member that `a` or `b`
// lacks is left out.
static int collect_fields(ssb200_canopy_flux *o, const ssb200_canopy_flux *a, const ssb200_canopy_flux *b,
                          FieldList &fl, bool with_sunlit, bool with_layers = true) {
  fl.n = 0;
  for (const ssb::FluxMember &m : ssb::kFluxMembers) {
    double *p = o->*m.ptr;
    const double *pa = a ? a->*m.ptr : nullptr, *pb = b ? b->*m.ptr : nullptr;
    if (!p || (!m.spectral && !with_sunlit) || (m.per_layer && !with_layers) || (a && (!pa || !pb))) continue;
    fl.p[fl.n] = p;
    fl.a[fl.n] = pa;
    fl.b[fl.n] = pb;
    fl.per_layer[fl.n] = m.per_layer;
    fl.spectral[fl.n] = m.spectral;
    ++fl.n;
  }
  return fl.n;
}

// Packed layers [l0, l1) of the non-Flat columns in [c0, c1) (0-based).  contiguous: the layers of each
// such column follow those of the previous one.  ok = false: some column's layers lie outside
// 1..ntotlay (that column is left out of the range).
struct LayerSpan {
  size_t l0 = 0, l1 = 0;
  bool contiguous = true, ok = true;
};
LayerSpan layer_span(const ssb200_canopy_properties &cp, size_t c0, size_t c1) {
  LayerSpan r;
  const size_t ntot = (size_t)cp.ntotlay;
  size_t lo = ntot, hi = 0, expect = 0;
  bool first = true;
  for (size_t j = c0; j < c1; ++j) {
    if (cp.i_representation[j] == SSB200_TILE_FLAT || cp.nlay[j] <= 0) continue;
    const size_t s = (size_t)cp.istartlay[j] - 1, e = s + (size_t)cp.nlay[j];
    if (cp.istartlay[j] < 1 || e > ntot) {
      r.ok = false;
      continue;
    }
    if (!first && s != expect) r.contiguous = false;
    first = false;
    expect = e;
    lo = std::min(lo, s);
    hi = std::max(hi, e);
  }
  if (hi > lo) {
    r.l0 = lo;
    r.l1 = hi;
  }
  return r;
}

// What the driver sequence derives for the members the caller leaves NULL: read_input's defaults and
// sigma T^4 emission from the temperatures.  Both driver-sequence entries plan it here; each launches
// fill() over the call's layers and derive() per column window of its own schedule.
struct DriverStage {
  struct Fill {  // constant, per packed layer
    double *p;
    double v;
    size_t width;
  };
  struct Emis {  // out = sigma [emissivity] T^4, interval 1
    double *out;
    const double *emissivity, *temperature;
    bool per_layer;
  };
  std::vector<Fill> fills;
  std::vector<Emis> emis;
  double *vcf = nullptr;  // default veg_contact_fraction (per packed layer)

  // Points the NULL members of the device-array structs cp / sw / lw at buffers of `pool`.  The
  // temperatures of `emis` are those of `drv`.  Returns 0 or a negative SSB200_ERR_* code.
  int plan(const ssb200_config &cfg, const ssb200_driver_inputs &drv, size_t ncol, size_t ntot,
           ssb200_canopy_properties &cp, ssb200_sw_spectral_properties &sw, ssb200_lw_spectral_properties &lw,
           Pool &pool) {
    if (!cp.veg_contact_fraction && cp.veg_fraction && cp.building_fraction) {
      vcf = pool.get<double>(ntot);  // driver/spartacus_surface_read_input.F90:155-166
      cp.veg_contact_fraction = vcf;
    }
    auto filled = [&](const double *&slot, size_t width, double v) {
      slot = pool.get<double>(ntot * width);
      fills.push_back(Fill{const_cast<double *>(slot), v, width});
    };
    if (cfg.do_sw) {  // driver/spartacus_surface_read_input.F90:258-269,335-344 (roof_albedo_dir NULL: the kernels use roof_albedo)
      const size_t g = (size_t)cfg.nsw;
      if (!sw.air_ext) filled(sw.air_ext, g, 1.0e-5);
      if (!sw.air_ssa) filled(sw.air_ssa, g, 0.999);
      if (!sw.wall_specular_frac && sw.wall_albedo) filled(sw.wall_specular_frac, g, 0.0);
    }
    if (cfg.do_lw) {  // driver/spartacus_surface_read_input.F90:362-365; radsurf_simple_spectrum.F90:41-66
      const size_t g = (size_t)cfg.nlw;
      if (!lw.air_ext) filled(lw.air_ext, g, 1.0e-5);
      if (!lw.air_ssa) filled(lw.air_ssa, g, 0.0);
      const bool need_t = !lw.ground_emission || !lw.roof_emission || !lw.wall_emission || !lw.clear_air_planck ||
                          !lw.veg_planck || !lw.veg_air_planck;
      if (need_t && g != 1)
        return fail(SSB200_ERR_ARG, "Simple longwave spectrum only possible with one input spectral interval");
      auto emission = [&](const double *&slot, const double *emissivity, const double *t, bool per_layer) {
        if (slot || !t) return;
        slot = pool.get<double>(per_layer ? ntot : ncol);
        emis.push_back(Emis{const_cast<double *>(slot), emissivity, t, per_layer});
      };
      emission(lw.ground_emission, lw.ground_emissivity, drv.ground_temperature, false);
      emission(lw.roof_emission, lw.roof_emissivity, drv.roof_temperature, true);
      emission(lw.wall_emission, lw.wall_emissivity, drv.wall_temperature, true);
      emission(lw.clear_air_planck, nullptr, drv.clear_air_temperature, true);
      emission(lw.veg_planck, nullptr, drv.veg_temperature, true);
      emission(lw.veg_air_planck, nullptr, drv.veg_air_temperature, true);
    }
    return pool.rc;
  }
  void fill(size_t l0, size_t l1, cudaStream_t st) const {
    for (const Fill &f : fills) {
      const long i0 = (long)(l0 * f.width), i1 = (long)(l1 * f.width);
      if (i1 <= i0) continue;
      k_fill<<<(unsigned)((i1 - i0 + 255) / 256), 256, 0, st>>>(f.p, f.v, i0, i1);
      ++g_launches;
    }
  }
  // default contact fraction and emission of columns [c0, c1) and packed layers [l0, l1); cp: the
  // caller's device arrays.  f32: the fractions, temperatures and emissivities read here are float
  // (ssb200_radsurf_fluxes_device_sp); the results stay FP64 either way.
  void derive(const ssb200_canopy_properties &cp, double min_veg, size_t c0, size_t c1, size_t l0, size_t l1,
              cudaStream_t st, bool f32 = false) const {
    if (f32)
      derive_as<float>(cp, min_veg, c0, c1, l0, l1, st);
    else
      derive_as<double>(cp, min_veg, c0, c1, l0, l1, st);
  }
  // the buffers of the plan: double whatever the precision of the caller's arrays
  std::vector<const void *> buffers() const {
    std::vector<const void *> v;
    if (vcf) v.push_back(vcf);
    for (const Fill &f : fills) v.push_back(f.p);
    for (const Emis &e : emis) v.push_back(e.out);
    return v;
  }

 private:
  template <class T>
  void derive_as(const ssb200_canopy_properties &cp, double min_veg, size_t c0, size_t c1, size_t l0, size_t l1,
                 cudaStream_t st) const {
    if (vcf && l1 > l0) {
      k_vcf_default<T><<<(unsigned)((l1 - l0 + 255) / 256), 256, 0, st>>>(
          vcf, (const T *)cp.veg_fraction, (const T *)cp.building_fraction, min_veg, (long)l0, (long)l1);
      ++g_launches;
    }
    for (const Emis &e : emis) {
      const long i0 = (long)(e.per_layer ? l0 : c0), i1 = (long)(e.per_layer ? l1 : c1);
      if (i1 <= i0) continue;
      k_sigma_t4<T><<<(unsigned)((i1 - i0 + 255) / 256), 256, 0, st>>>(e.out, (const T *)e.emissivity,
                                                                         (const T *)e.temperature, 1, i0, i1);
      ++g_launches;
    }
  }
};

// widen every array of `v` (round = false) or round its outputs back (true) on `st`, kConvMax arrays per launch
int convert_arrays(const std::vector<ConvArray> &v, bool round, cudaStream_t st) {
  ConvList cl;
  cl.n = 0;
  long most = 0;
  auto flush = [&]() -> int {
    if (cl.n > 0 && most > 0) {
      const unsigned blocks = (unsigned)((most + 255) / 256);
      if (round)
        k_convert<true><<<blocks, 256, 0, st>>>(cl);
      else
        k_convert<false><<<blocks, 256, 0, st>>>(cl);
      ++g_launches;
      SSB_CUDA(cudaGetLastError());
    }
    cl.n = 0;
    most = 0;
    return 0;
  };
  for (const ConvArray &c : v) {
    if ((round && !c.out) || c.hi <= c.lo) continue;
    cl.f[cl.n] = c.f;
    cl.d[cl.n] = c.d;
    cl.lo[cl.n] = c.lo;
    cl.hi[cl.n] = c.hi;
    ++cl.n;
    most = std::max(most, c.hi - c.lo);
    if (cl.n == kConvMax)
      if (int rc = flush()) return rc;
  }
  return flush();
}

// --- host-pointer staging --------------------------------------------------
struct Stager {
  Pool pool;  // device mirrors and device-only arrays of the call
  struct Arr {
    double *host;    // (sp: really float *)
    double *dev;
    float *dev32;    // sp: device copy in the caller's precision
    size_t width;    // doubles per column (per_layer = false) or per packed layer (true)
    bool per_layer, upload, download;
  };
  std::vector<Arr> arrs;
  // single-precision storage (ssb200_radsurf_sp): the caller's arrays hold float; they cross PCIe as
  // float and are widened / rounded on the device, the kernels see double mirrors as always
  bool sp = false;
  Stager(Context &c, bool sp_) : pool{c.stage, "staging allocation: "}, sp(sp_) {}
  // device mirror of `host` (total = rows * width doubles); copies are issued per window
  double *mirror(const double *host, size_t rows, size_t width, bool per_layer, bool upload, bool download) {
    if (!host) return nullptr;
    double *dev = pool.get<double>(rows * width);
    float *dev32 = sp ? pool.get<float>(rows * width) : nullptr;
    if (pool.rc) return nullptr;
    arrs.push_back(Arr{const_cast<double *>(host), dev, dev32, width, per_layer, upload, download});
    return dev;
  }
  // copy the slices of columns [c0, c1) / packed layers [l0, l1) on stream `st`
  int copy_window(bool to_device, size_t c0, size_t c1, size_t l0, size_t l1, cudaStream_t st) {
    for (const Arr &a : arrs) {
      if (to_device ? !a.upload : !a.download) continue;
      const size_t off = (a.per_layer ? l0 : c0) * a.width, cnt = ((a.per_layer ? l1 : c1) * a.width) - off;
      if (cnt == 0) continue;
      cudaError_t e;
      if (sp) {
        float *h32 = reinterpret_cast<float *>(a.host);
        const unsigned blocks = (unsigned)((cnt + 255) / 256);
        if (to_device) {
          e = cudaMemcpyAsync(a.dev32 + off, h32 + off, cnt * sizeof(float), cudaMemcpyHostToDevice, st);
          k_f2d<<<blocks, 256, 0, st>>>(a.dev + off, a.dev32 + off, cnt);
        } else {
          k_d2f<<<blocks, 256, 0, st>>>(a.dev32 + off, a.dev + off, cnt);
          e = cudaMemcpyAsync(h32 + off, a.dev32 + off, cnt * sizeof(float), cudaMemcpyDeviceToHost, st);
        }
        ++g_launches;
        if (e == cudaSuccess) e = cudaGetLastError();
      } else {
        e = to_device ? cudaMemcpyAsync(a.dev + off, a.host + off, cnt * sizeof(double), cudaMemcpyHostToDevice, st)
                      : cudaMemcpyAsync(a.host + off, a.dev + off, cnt * sizeof(double), cudaMemcpyDeviceToHost, st);
      }
      if (e != cudaSuccess)
        return fail(SSB200_ERR_CUDA, std::string(to_device ? "H2D copy: " : "D2H copy: ") + cudaGetErrorString(e));
    }
    return 0;
  }
};

}  // namespace

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

const char *ssb200_version(void) { return "spartacus_surface_b200 0.1 (sm_100a, generic + register-resident kernels)"; }

const char *ssb200_last_error(void) { return g_last_error.c_str(); }

int ssb200_abi_sizes(int64_t out[7]) {
  if (!out) return fail(SSB200_ERR_ARG, "NULL argument");
  out[0] = sizeof(ssb200_legendre_gauss);
  out[1] = sizeof(ssb200_config);
  out[2] = sizeof(ssb200_canopy_properties);
  out[3] = sizeof(ssb200_sw_spectral_properties);
  out[4] = sizeof(ssb200_lw_spectral_properties);
  out[5] = sizeof(ssb200_canopy_flux);
  out[6] = sizeof(ssb200_boundary_conds_out);
  return 0;
}

int ssb200_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int ssb200_set_device(int device) {
  int rc = ensure_device();
  if (rc) return rc;
  SSB_CUDA(cudaSetDevice(device));
  return 0;
}

// legendre_gauss_type%initialize (radtool/radtool_legendre_gauss.F90:52-100,119-170):
// Newton iteration for the Legendre nodes mapped to [0,1]; host side, once per config.
int ssb200_legendre_gauss_init(int32_t nstream, ssb200_legendre_gauss *lg) {
  if (!lg || nstream < 1 || nstream > SSB200_MAX_NSTREAM) return fail(SSB200_ERR_ARG, "nstream outside 1..16");
  const int n = nstream;
  const double pi = SSB_PI, eps = SSB_EPS;
  double y[SSB200_MAX_NSTREAM], y0[SSB200_MAX_NSTREAM], dp[SSB200_MAX_NSTREAM];
  double P[SSB200_MAX_NSTREAM + 1][SSB200_MAX_NSTREAM];
  const float c027 = 0.27f / (float)n;  // single-precision constant expression in the reference (:142)
  for (int k = 1; k <= n; ++k) {
    y[k - 1] = cos((2 * (k - 1) + 1) * pi / (2 * n)) + (double)c027 * sin(pi * (-1.0 + 2.0 * k) / (n + 1));
    y0[k - 1] = 2.0;
  }
  for (;;) {
    double md = 0.0;
    for (int i = 0; i < n; ++i) md = fmax(md, fabs(y[i] - y0[i]));
    if (!(md > eps)) break;
    for (int i = 0; i < n; ++i) {
      P[0][i] = 1.0;
      P[1][i] = y[i];
    }
    for (int k = 2; k <= n; ++k)
      for (int i = 0; i < n; ++i) P[k][i] = ((2 * k - 1) * y[i] * P[k - 1][i] - (k - 1) * P[k - 2][i]) / k;
    for (int i = 0; i < n; ++i) dp[i] = (n + 1) * (P[n - 1][i] - y[i] * P[n][i]) / (1.0 - y[i] * y[i]);
    for (int i = 0; i < n; ++i) {
      y0[i] = y[i];
      y[i] = y0[i] - P[n][i] / dp[i];
    }
  }
  memset(lg, 0, sizeof(*lg));
  lg->nstream = n;
  double sh = 0.0, sv = 0.0, s2 = 0.0;
  for (int i = 0; i < n; ++i) {
    lg->mu[i] = 0.5 * (0.0 * (1.0 - y[i]) + 1.0 * (1.0 - y[i]));  // map as written in the reference (:165)
    lg->weight[i] = (((n + 1) * (n + 1)) / (double)(n * n)) * (1.0 - 0.0) / ((1.0 - y[i] * y[i]) * dp[i] * dp[i]);
    lg->sin_ang[i] = sqrt(1.0 - lg->mu[i] * lg->mu[i]);
    lg->tan_ang[i] = lg->sin_ang[i] / lg->mu[i];
    lg->hweight[i] = lg->weight[i] * lg->mu[i];
    lg->vweight[i] = lg->weight[i] * lg->sin_ang[i];
  }
  for (int i = 0; i < n; ++i) {
    sh += lg->hweight[i];
    sv += lg->vweight[i];
  }
  for (int i = 0; i < n; ++i) {
    lg->hweight[i] = lg->hweight[i] / sh;
    lg->vweight[i] = lg->vweight[i] / sv;
  }
  lg->vadjustment = 1.0;
  for (int i = 0; i < n; ++i) s2 += lg->weight[i] * lg->sin_ang[i];
  lg->vadjustment2 = (pi / 4.0) / s2;
  return 0;
}

int ssb200_radsurf_device(const ssb200_config *config, const ssb200_canopy_properties *canopy_props,
                          const ssb200_sw_spectral_properties *sw, const ssb200_lw_spectral_properties *lw,
                          ssb200_boundary_conds_out *bc_out, int32_t istartcol, int32_t iendcol,
                          ssb200_canopy_flux *sw_norm_dir, ssb200_canopy_flux *sw_norm_diff,
                          ssb200_canopy_flux *lw_internal, ssb200_canopy_flux *lw_norm, void *stream,
                          int32_t *status_out) {
  int rc = ensure_device();
  if (rc) return rc;
  std::lock_guard<std::mutex> lock(g_mutex);
  ssb::CallArgs ca{config, canopy_props, sw, lw, bc_out, sw_norm_dir, sw_norm_diff, lw_internal, lw_norm};
  return radsurf_device_locked(g_ctx, ca, istartcol, iendcol, (cudaStream_t)stream, status_out);
}

// Body of ssb200_radsurf_device_sp: every real array of `ca` is a float device array.  The per-column
// members (cos_sza, ground_*, bc_out, the per-column flux members: 1/16 of the data at 16 layers) are
// widened into double buffers of the context for the call's columns and rounded back after the solve.
// The per-layer members take one of two routes, chosen per call from the plan:
//   staged:   every class and pass reads and writes them through the level-major staging only, whose
//             gather widens (float -> double) and whose scatter rounds (double -> float): no double copy;
//   fallback: some read happens outside the staging (generic kernels, stage_layers = 0, column-resident
//             kernels, single-layer urban columns on the surface kernel): the packed layers of the call's
//             columns are widened into double copies and rounded back, as ssb200_radsurf_sp does.
// Either way the kernels see the doubles the double entry sees on widened inputs, and entries the
// solve leaves untouched round back to the caller's value.
static int radsurf_device_sp_locked(Context &cx, const ssb::CallArgs &ca, int32_t istartcol, int32_t iendcol,
                                    cudaStream_t stream, int32_t *status_out) {
  int range[2] = {1, 0};
  int rc = radsurf_device_locked(cx, ca, istartcol, iendcol, stream, nullptr, range);
  if (rc || range[0] > range[1]) return rc;
  const ssb200_config &cfg = *ca.config;
  const ssb200_canopy_properties &cp = *ca.cp;
  CudaBackend probe(cx);
  ssb::Dispatcher<CudaBackend> route(probe);
  const bool staged = route.all_layers_staged(ca, cx.plan);
  const size_t ncol = (size_t)cp.ncol, ntot = (size_t)cp.ntotlay;
  const size_t c0 = (size_t)range[0] - 1, c1 = (size_t)range[1];
  LayerSpan span;  // packed layers of the call's columns (fallback route)
  if (!staged) span = layer_span(cp, c0, c1);
  std::vector<ConvArray> conv;
  Pool pool{cx.wide, "double copies: "};
  // double buffer for the float array p of `rows` x `width` values; rows [r0, r1) are converted
  auto wide = [&](const void *p, size_t rows, size_t width, size_t r0, size_t r1, bool out) -> double * {
    if (!p) return nullptr;
    double *d = pool.get<double>(rows * width);
    if (d) conv.push_back(ConvArray{(float *)p, d, (long)(r0 * width), (long)(r1 * width), out});
    return d;
  };
  // the members of `d` as the kernels see them: per-column members widened over the call's columns,
  // per-layer members passed to the staging (staged route) or widened over the call's layers
  auto widen = [&](auto &d, const auto &table, size_t nspec, bool out) {
    for (const auto &m : table) {
      const size_t w = ssb::member_width(m, nspec);
      const void *p = d.*m.ptr;
      d.*m.ptr = !m.per_layer ? wide(p, ncol, w, c0, c1, out)
                              : staged ? (double *)p : wide(p, ntot, w, span.l0, span.l1, out);
    }
  };
  ssb200_canopy_properties dcp = cp;
  widen(dcp, ssb::kCanopyMembers, 1, false);
  ssb200_sw_spectral_properties dsw;
  ssb200_lw_spectral_properties dlw;
  ssb200_boundary_conds_out dbc;
  memset(&dsw, 0, sizeof(dsw));
  memset(&dlw, 0, sizeof(dlw));
  memset(&dbc, 0, sizeof(dbc));
  if (cfg.do_sw) {
    dsw = *ca.sw;
    widen(dsw, ssb::kSwMembers, (size_t)cfg.nsw, false);
  }
  if (cfg.do_lw) {
    dlw = *ca.lw;
    widen(dlw, ssb::kLwMembers, (size_t)cfg.nlw, false);
  }
  for (const ssb::BcMember &m : ssb::kBcMembers)
    if (m.lw ? cfg.do_lw : cfg.do_sw)
      dbc.*m.ptr = wide(ca.bc->*m.ptr, ncol, (size_t)(m.lw ? cfg.nlw : cfg.nsw), c0, c1, true);
  auto flux = [&](const ssb200_canopy_flux *h, ssb200_canopy_flux &d) {
    d = *h;
    widen(d, ssb::kFluxMembers, (size_t)h->nspec, true);
  };
  ssb200_canopy_flux d1, d2, d3, d4;
  if (cfg.do_sw) {
    flux(ca.sw_dir, d1);
    flux(ca.sw_diff, d2);
  }
  if (cfg.do_lw) {
    flux(ca.lw_int, d3);
    flux(ca.lw_norm, d4);
  }
  if (pool.rc) return pool.rc;
  ssb::CallArgs wca{ca.config, &dcp, cfg.do_sw ? &dsw : nullptr, cfg.do_lw ? &dlw : nullptr, &dbc,
                    cfg.do_sw ? &d1 : nullptr, cfg.do_sw ? &d2 : nullptr,
                    cfg.do_lw ? &d3 : nullptr, cfg.do_lw ? &d4 : nullptr};
  Drain drain{stream};
  if ((rc = convert_arrays(conv, false, stream))) return rc;
  ssb::StagePrecision prec;
  prec.f32 = staged;
  if ((rc = dispatch_call(cx, wca, prec))) return rc;
  if ((rc = convert_arrays(conv, true, stream))) return rc;
  drain.armed = false;
  return finish_device_call(cx, stream, status_out);
}

// Body of ssb200_radsurf_fluxes_device and, with sp, ssb200_radsurf_fluxes_device_sp: the sequence of
// radsurf_host with drv != NULL on device arrays.  Inputs the caller leaves NULL are filled in context
// buffers (read_input's defaults, sigma T^4 from the temperatures) over the call's columns and packed layers.
// The four normalised flux objects take one of two routes, chosen per call from the plan:
//   staged:   every per-layer write goes through the level-major staging, whose scatter writes
//             fa * f1 + fb * f2 straight into sw_flux / lw_flux (StageList::sum): the per-layer members of
//             the normalised objects exist in the staging buffers of a chunk only.  Their per-column
//             members (written in place by the sweeps and the surface kernel) live in zeroed context
//             buffers and are scaled and summed by one launch per pass after the solve;
//   fallback: generic kernels, stage_layers = 0, column-resident kernels, single-layer urban columns:
//             the four objects are materialised in zeroed context buffers for the call's columns and
//             layers, and scaled and summed per column and per owned layer after the solve.
// Both give the bits of ssb200_radsurf_fluxes: the same products and sums, each rounded once.
// sp: every real array of the caller, driver_inputs included, holds float.  The defaults, the emission
// and the default contact fraction stay in double context buffers, computed from the float inputs widened
// exactly.  The caller's per-column members, bc_out and the top-of-canopy fluxes are widened into context
// buffers for the call's columns (bc_out is rounded back after the solve).  On the staged route the
// staging widens the caller's per-layer inputs and its summing scatter rounds into the float summed
// objects; on the fallback route the per-layer inputs are widened over the call's layers.  Either way the
// scale + sum rounds the FP64 result once into the summed objects, so every output is the double entry's
// on widened inputs, rounded to nearest.
static int radsurf_fluxes_device_locked(Context &cx, const ssb200_config *config, const ssb200_canopy_properties *cp,
                                        const ssb200_sw_spectral_properties *sw, const ssb200_lw_spectral_properties *lw,
                                        const ssb200_driver_inputs *drv, ssb200_boundary_conds_out *bc,
                                        int32_t istartcol, int32_t iendcol, ssb200_canopy_flux *sw_flux,
                                        ssb200_canopy_flux *lw_flux, cudaStream_t stream, int32_t *status_out,
                                        bool sp = false) {
  const char *name = sp ? "radsurf_fluxes_device_sp" : "radsurf_fluxes_device";
  if (!config || !cp || !bc || !drv)
    return fail(SSB200_ERR_ARG, "config, canopy_props, driver_inputs and bc_out must not be NULL");
  if ((config->do_sw && (!sw_flux || !drv->top_flux_dn_sw || !drv->top_flux_dn_direct_sw)) ||
      (config->do_lw && (!lw_flux || !drv->top_flux_dn_lw)))
    return fail(SSB200_ERR_ARG, std::string(name) + ": flux object or top-of-canopy flux missing");
  {
    ssb::CallArgs probe{config, cp, sw, lw, bc, sw_flux, sw_flux, lw_flux, lw_flux};
    std::string err;
    const int rc = ssb::validate_call(probe, err);
    if (rc) return fail(rc, err);
  }
  const size_t ncol = (size_t)cp->ncol, ntot = (size_t)cp->ntotlay;
  int c1 = istartcol > 0 ? istartcol : 1, c2 = iendcol > 0 ? iendcol : cp->ncol;
  if (c2 > cp->ncol) c2 = cp->ncol;
  if (c1 > c2) return 0;
  const size_t c0 = (size_t)c1 - 1, cN = (size_t)c2;  // 0-based column window [c0, cN)
  // packed layers [l0, lN) spanned by the call's columns (ranges outside 1..ntotlay are refused by the plan)
  const LayerSpan span = layer_span(*cp, c0, cN);
  const size_t l0 = span.l0, lN = span.l1;
  Pool pool{cx.drv, "context buffers: "};
  ssb200_canopy_properties dcp = *cp;
  ssb200_sw_spectral_properties dsw;
  ssb200_lw_spectral_properties dlw;
  ssb200_boundary_conds_out dbc = *bc;
  memset(&dsw, 0, sizeof(dsw));
  memset(&dlw, 0, sizeof(dlw));
  if (config->do_sw) dsw = *sw;
  if (config->do_lw) dlw = *lw;
  DriverStage ds;
  int rc = ds.plan(*config, *drv, ncol, ntot, dcp, dsw, dlw, pool);
  if (rc) return rc;
  // plan, argument checks, ordering against the previous call, status reset (the summed objects stand in
  // for the normalised ones, whose shape they have)
  ssb::CallArgs ca{config, &dcp, config->do_sw ? &dsw : nullptr, config->do_lw ? &dlw : nullptr, &dbc,
                   sw_flux, sw_flux, lw_flux, lw_flux};
  int range[2] = {1, 0};
  rc = radsurf_device_locked(cx, ca, c1, c2, stream, nullptr, range);
  if (rc || range[0] > range[1]) return rc;
  CudaBackend probe(cx);
  ssb::Dispatcher<CudaBackend> route(probe);
  const bool staged = route.all_layers_staged(ca, cx.plan);
  ssb::StagePrecision prec;  // (the staging reaches the caller's float arrays on the staged route only)
  prec.f32 = sp && staged;
  prec.f64 = ds.buffers();
  // sp: double copies of the caller's float arrays, widened over rows [r0, r1) before the solve; `out`
  // ones (bc_out) are rounded back after it
  std::vector<ConvArray> conv;
  auto wide = [&](const void *p, size_t rows, size_t width, size_t r0, size_t r1, bool out) -> double * {
    if (!p) return nullptr;
    double *d = pool.get<double>(rows * width);
    if (d) conv.push_back(ConvArray{(float *)p, d, (long)(r0 * width), (long)(r1 * width), out});
    return d;
  };
  // the caller's members of `d`: per-column ones over the call's columns; per-layer ones over its layers on
  // the fallback route (the staging widens them on the staged route).  DriverStage's buffers are double.
  auto widen = [&](auto &d, const auto &table, size_t nspec) {
    for (const auto &m : table) {
      auto &member = d.*m.ptr;
      if (!member || (m.per_layer && staged)) continue;
      if (std::find(prec.f64.begin(), prec.f64.end(), (const void *)member) != prec.f64.end()) continue;
      const size_t w = ssb::member_width(m, nspec);
      member = m.per_layer ? wide(member, ntot, w, l0, lN, false) : wide(member, ncol, w, c0, cN, false);
    }
  };
  const double *top_sw = drv->top_flux_dn_sw, *top_dir = drv->top_flux_dn_direct_sw, *top_lw = drv->top_flux_dn_lw;
  if (sp) {
    widen(dcp, ssb::kCanopyMembers, 1);
    if (config->do_sw) widen(dsw, ssb::kSwMembers, (size_t)config->nsw);
    if (config->do_lw) widen(dlw, ssb::kLwMembers, (size_t)config->nlw);
    for (const ssb::BcMember &m : ssb::kBcMembers)
      dbc.*m.ptr = (m.lw ? config->do_lw : config->do_sw)
                       ? wide(bc->*m.ptr, ncol, (size_t)(m.lw ? config->nlw : config->nsw), c0, cN, true)
                       : nullptr;
    if (config->do_sw) {
      top_sw = wide(top_sw, ncol, (size_t)config->nsw, c0, cN, false);
      top_dir = wide(top_dir, ncol, (size_t)config->nsw, c0, cN, false);
    }
    if (config->do_lw) top_lw = wide(top_lw, ncol, (size_t)config->nlw, c0, cN, false);
  }
  // the normalised objects: context buffers shaped like the summed object, zeroed over the call's window
  // (canopy_flux_type%zero_all, driver:184).  Staged route: per-column members only; the per-layer members
  // keep the summed object's pointers, which only mark them present (stage_plan redirects them).
  std::vector<std::pair<double *, size_t>> zeroed;
  auto normalised = [&](const ssb200_canopy_flux *sum, ssb200_canopy_flux &d) {
    d = *sum;
    for (const ssb::FluxMember &m : ssb::kFluxMembers) {
      double *&member = d.*m.ptr;
      if (!member || (m.per_layer && staged)) continue;
      const size_t w = ssb::member_width(m, (size_t)sum->nspec);
      member = pool.get<double>((m.per_layer ? ntot : ncol) * w);
      if (member) zeroed.push_back({member + (m.per_layer ? l0 : c0) * w, (m.per_layer ? lN - l0 : cN - c0) * w});
    }
  };
  ssb200_canopy_flux d1, d2, d3, d4;
  PassSum sum_sw, sum_lw;
  if (config->do_sw) {
    normalised(sw_flux, d1);
    normalised(sw_flux, d2);
    sum_sw.fa = top_dir;
    sum_sw.fb = top_sw;
    sum_sw.fb_minus = top_dir;
    if (staged) sum_sw.out = sw_flux;
  }
  if (config->do_lw) {
    normalised(lw_flux, d3);
    normalised(lw_flux, d4);
    sum_lw.fb = top_lw;
    if (staged) sum_lw.out = lw_flux;
  }
  if (pool.rc) return pool.rc;
  const ssb::CallArgs nca{config, &dcp, ca.sw, ca.lw, &dbc, config->do_sw ? &d1 : nullptr, config->do_sw ? &d2 : nullptr,
                          config->do_lw ? &d3 : nullptr, config->do_lw ? &d4 : nullptr};
  Drain drain{stream};
  CudaBackend be(cx);  // (profiling: the stages around the solve are booked with family 4)
  be.tick(4, true);
  if ((rc = convert_arrays(conv, false, stream))) return rc;
  ds.fill(l0, lN, stream);
  ds.derive(*cp, config->min_vegetation_fraction, c0, cN, l0, lN, stream, sp);
  for (const auto &z : zeroed)
    if (z.second > 0) SSB_CUDA(cudaMemsetAsync(z.first, 0, z.second * sizeof(double), stream));
  SSB_CUDA(cudaGetLastError());
  be.tick(4, false);
  if ((rc = dispatch_call(cx, nca, prec, sum_sw, sum_lw))) return rc;
  // scale + sum (driver:250-261) of what the solve left in the normalised objects: the per-column members
  // (staged route), or every member over the call's columns and owned layers (fallback route), rounded
  // once into float summed objects (sp)
  if (!staged && (rc = ensure_lay2col(cx, ncol, ntot, stream))) return rc;
  const long cnt = (long)std::max(cN - c0, staged ? (size_t)0 : lN - l0);
  auto scale_sum = [&](ssb200_canopy_flux *o, const ssb200_canopy_flux &x, const ssb200_canopy_flux &y,
                       const double *fa, const double *fb, const double *fbm, int nspec) {
    FieldList fl;
    collect_fields(o, &x, &y, fl, true, !staged);
    const long nthr = cnt * nspec;
    if (fl.n == 0 || nthr <= 0) return;
    const unsigned blocks = (unsigned)((nthr + 255) / 256);
    const int *lay2col = (const int *)cx.d_lay2col.p;
    if (sp)
      k_scale_sum<float><<<blocks, 256, 0, stream>>>(fl, fa, fb, fbm, lay2col, nspec, (long)c0, (long)cN, (long)l0, (long)lN);
    else
      k_scale_sum<double><<<blocks, 256, 0, stream>>>(fl, fa, fb, fbm, lay2col, nspec, (long)c0, (long)cN, (long)l0, (long)lN);
    ++g_launches;
  };
  be.tick(4, true);
  if (config->do_sw) scale_sum(sw_flux, d1, d2, sum_sw.fa, sum_sw.fb, sum_sw.fb_minus, config->nsw);
  if (config->do_lw) scale_sum(lw_flux, d3, d4, nullptr, sum_lw.fb, nullptr, config->nlw);
  SSB_CUDA(cudaGetLastError());
  if ((rc = convert_arrays(conv, true, stream))) return rc;
  be.tick(4, false);
  drain.armed = false;
  return finish_device_call(cx, stream, status_out);
}

// Body of both host entries.  drv == NULL: ssb200_radsurf (the four normalised flux objects are
// host arrays).  drv != NULL: ssb200_radsurf_fluxes - the normalised objects exist on the device
// only (shaped like sw_flux / lw_flux), NULL inputs take read_input's defaults or are derived from
// the temperatures, and every window ends with the fused scale + sum into sw_flux / lw_flux.
static int radsurf_host(const ssb200_config *config, const ssb200_canopy_properties *cp,
                        const ssb200_sw_spectral_properties *sw, const ssb200_lw_spectral_properties *lw,
                        const ssb200_driver_inputs *drv, ssb200_boundary_conds_out *bc, int32_t istartcol,
                        int32_t iendcol, ssb200_canopy_flux *sw_dir, ssb200_canopy_flux *sw_diff,
                        ssb200_canopy_flux *lw_int, ssb200_canopy_flux *lw_norm, ssb200_canopy_flux *sw_flux,
                        ssb200_canopy_flux *lw_flux, bool sp = false) {
  int rc = ensure_device();
  if (rc) return rc;
  std::lock_guard<std::mutex> lock(g_mutex);
  Context &cx = g_ctx;
  if (!config || !cp || !bc) return fail(SSB200_ERR_ARG, "config, canopy_props and bc_out must not be NULL");
  if (drv) {
    if ((config->do_sw && (!sw_flux || !drv->top_flux_dn_sw || !drv->top_flux_dn_direct_sw)) ||
        (config->do_lw && (!lw_flux || !drv->top_flux_dn_lw)))
      return fail(SSB200_ERR_ARG, "radsurf_fluxes: flux object or top-of-canopy flux missing");
    sw_dir = sw_diff = sw_flux;  // shape donors for the argument checks
    lw_int = lw_norm = lw_flux;
  }
  {
    ssb::CallArgs probe{config, cp, sw, lw, bc, sw_dir, sw_diff, lw_int, lw_norm};
    std::string err;
    rc = ssb::validate_call(probe, err);
    if (rc) return fail(rc, err);
  }
  if (!cx.own_stream) SSB_CUDA(cudaStreamCreateWithFlags(&cx.own_stream, cudaStreamNonBlocking));
  cudaStream_t st = cx.own_stream;
  int c1 = istartcol > 0 ? istartcol : 1, c2 = iendcol > 0 ? iendcol : cp->ncol;
  if (c2 > cp->ncol) c2 = cp->ncol;
  if (c1 > c2) return 0;
  const size_t ncol = (size_t)cp->ncol, ntot = (size_t)cp->ntotlay;
  // packed layer range touched by the columns of this call: per-layer outputs need no upload when it is
  // contiguous
  const LayerSpan span = layer_span(*cp, (size_t)c1 - 1, (size_t)c2);
  if (!span.ok) return fail(SSB200_ERR_SHAPE, "layer range outside 1..ntotlay");
  const bool contiguous = span.contiguous;
  const size_t l1 = span.l0, l2 = span.l1, cN = (size_t)(c2 - c1 + 1), lN = l2 - l1;
  if (drv && !contiguous)
    return fail(SSB200_ERR_UNSUPPORTED, "radsurf_fluxes needs the packed layers of the selected columns to be contiguous");
  Stager sg(cx, sp);
  // inputs: mirrors uploaded per window
  auto inputs = [&](auto &d, const auto &h, const auto &table, size_t nspec) {
    d = h;
    for (const auto &m : table)
      d.*m.ptr = sg.mirror(h.*m.ptr, m.per_layer ? ntot : ncol, ssb::member_width(m, nspec), m.per_layer, true, false);
  };
  ssb200_canopy_properties dcp;
  ssb200_sw_spectral_properties dsw;
  ssb200_lw_spectral_properties dlw;
  memset(&dsw, 0, sizeof(dsw));
  memset(&dlw, 0, sizeof(dlw));
  inputs(dcp, *cp, ssb::kCanopyMembers, 1);
  if (config->do_sw) inputs(dsw, *sw, ssb::kSwMembers, (size_t)config->nsw);
  if (config->do_lw) inputs(dlw, *lw, ssb::kLwMembers, (size_t)config->nlw);
  // read_input's defaults and the emission for members the caller leaves NULL (ssb200_radsurf_fluxes only)
  DriverStage ds;
  if (drv) {
    if (sg.pool.rc) return sg.pool.rc;
    if ((rc = ds.plan(*config, *drv, ncol, ntot, dcp, dsw, dlw, sg.pool))) return rc;
    // (the same host array given for several temperatures - the driver passes one air temperature
    // for clear air, vegetation and the air in vegetation - is uploaded once)
    std::vector<std::pair<const double *, const double *>> t_seen;
    for (DriverStage::Emis &e : ds.emis) {
      const double *h = e.temperature;
      e.temperature = nullptr;
      for (const auto &s : t_seen)
        if (s.first == h) e.temperature = s.second;
      if (!e.temperature) {
        e.temperature = sg.mirror(h, e.per_layer ? ntot : ncol, 1, e.per_layer, true, false);
        t_seen.push_back({h, e.temperature});
      }
    }
  }
  // outputs: per-column members are uploaded first (Flat tiles and night-time
  // columns leave some of them untouched); per-layer members are fully
  // rewritten by the kernels when the layer range is contiguous
  ssb200_boundary_conds_out dbc;
  memset(&dbc, 0, sizeof(dbc));
  for (const ssb::BcMember &m : ssb::kBcMembers)
    if (m.lw ? config->do_lw : config->do_sw)
      dbc.*m.ptr = sg.mirror(bc->*m.ptr, ncol, (size_t)(m.lw ? config->nlw : config->nsw), false, true, true);
  auto stage_flux = [&](const ssb200_canopy_flux *h, ssb200_canopy_flux &d) {
    d = *h;
    for (const ssb::FluxMember &m : ssb::kFluxMembers)
      d.*m.ptr = sg.mirror(h->*m.ptr, m.per_layer ? ntot : ncol, ssb::member_width(m, (size_t)h->nspec), m.per_layer,
                           !m.per_layer || !contiguous, true);
  };
  // a normalised flux object that lives on the device only, with the members of `tmpl`; members the
  // kernels may leave untouched start from zero (canopy_flux_type%zero_all, driver:184)
  std::vector<std::pair<double *, size_t>> zeroed;
  auto device_flux = [&](const ssb200_canopy_flux *tmpl, ssb200_canopy_flux &d) {
    d = *tmpl;
    for (const ssb::FluxMember &m : ssb::kFluxMembers) {
      double *&member = d.*m.ptr;
      if (!member) continue;
      const size_t total = (m.per_layer ? ntot : ncol) * ssb::member_width(m, (size_t)tmpl->nspec);
      member = sg.pool.get<double>(total);
      if (!m.per_layer || !contiguous) zeroed.push_back({member, total});
    }
  };
  ssb200_canopy_flux d1, d2, d3, d4, dsum_sw, dsum_lw;
  const double *d_top_sw = nullptr, *d_top_dir = nullptr, *d_top_lw = nullptr;
  if (drv) {
    if (config->do_sw) {
      device_flux(sw_flux, d1);
      device_flux(sw_flux, d2);
      stage_flux(sw_flux, dsum_sw);
      d_top_sw = sg.mirror(drv->top_flux_dn_sw, ncol, (size_t)config->nsw, false, true, false);
      d_top_dir = sg.mirror(drv->top_flux_dn_direct_sw, ncol, (size_t)config->nsw, false, true, false);
    }
    if (config->do_lw) {
      device_flux(lw_flux, d3);
      device_flux(lw_flux, d4);
      stage_flux(lw_flux, dsum_lw);
      d_top_lw = sg.mirror(drv->top_flux_dn_lw, ncol, (size_t)config->nlw, false, true, false);
    }
  } else {
    if (config->do_sw) {
      stage_flux(sw_dir, d1);
      stage_flux(sw_diff, d2);
    }
    if (config->do_lw) {
      stage_flux(lw_int, d3);
      stage_flux(lw_norm, d4);
    }
  }
  if (sg.pool.rc) return sg.pool.rc;
  ds.fill(l1, l2, st);
  for (const auto &z : zeroed) SSB_CUDA(cudaMemsetAsync(z.first, 0, z.second * sizeof(double), st));
  ssb::CallArgs ca{config, &dcp, config->do_sw ? &dsw : nullptr, config->do_lw ? &dlw : nullptr, &dbc,
                   config->do_sw ? &d1 : nullptr, config->do_sw ? &d2 : nullptr,
                   config->do_lw ? &d3 : nullptr, config->do_lw ? &d4 : nullptr};
  // Pipeline: the column range is cut into blocks whose input slices are uploaded, solved
  // and downloaded as three overlapping stages (pinned host memory needed for true
  // overlap).  Requires a contiguous packed-layer range; profiling serialises.
  int range[2];
  rc = radsurf_device_locked(cx, ca, c1, c2, st, nullptr, range);
  if (rc) return rc;
  if (drv && (rc = ensure_lay2col(cx, ncol, ntot, st))) return rc;
  SSB_CUDA(cudaStreamSynchronize(st));  // plan upload and status reset are visible to every lane
  const size_t total_work = lN + cN;
  int nblk = 1;
  if (cx.pipeline && contiguous && !cx.profiling && total_work >= ((size_t)1 << 17)) {
    // blocks of at least ~30 k columns x 16 layers: smaller launches are bound by launch latency (a rank
    // of an 8-GPU run holds 131,072 columns: 4 blocks, not 16)
    nblk = (int)(total_work >> 19);
    if (nblk < 2) nblk = 2;
    if (nblk > cx.pipeline_max_blocks) nblk = cx.pipeline_max_blocks;
  }
  // three stages on three streams, chained per block by events: uploads in block order on
  // lane 0, kernels on lane 1 (one scratch area with the full budget, reused block after
  // block), downloads on lane 2 - both copy engines stay busy once the pipeline has filled
  for (int l = 0; l < Context::kLanes; ++l)
    if (!cx.lane_stream[l]) SSB_CUDA(cudaStreamCreateWithFlags(&cx.lane_stream[l], cudaStreamNonBlocking));
  cudaStream_t s_up = cx.lane_stream[0], s_run = cx.lane_stream[1], s_down = cx.lane_stream[2];
  if (nblk == 1) s_up = s_down = s_run;
  if ((int)cx.blk_events.size() < 2 * nblk) {
    const size_t old_n = cx.blk_events.size();
    cx.blk_events.resize((size_t)2 * nblk, nullptr);
    for (size_t i = old_n; i < cx.blk_events.size(); ++i)
      SSB_CUDA(cudaEventCreateWithFlags(&cx.blk_events[i], cudaEventDisableTiming));
  }
  // first packed layer of every column >= j (Flat tiles own no layers): block boundaries
  auto layer_begin = [&](int j) -> size_t {
    for (; j < c2; ++j)
      if (cp->i_representation[j] != SSB200_TILE_FLAT && cp->nlay[j] > 0) return (size_t)cp->istartlay[j] - 1;
    return l2;
  };
  // an error return inside the loop must not leave queued copies reading / writing the caller's
  // host arrays after the function has returned (the caller may free them): drain the lanes first
  struct LaneDrain {
    Context &cx;
    bool armed = true;
    ~LaneDrain() {
      if (armed)
        for (int l = 0; l < Context::kLanes; ++l) cudaStreamSynchronize(cx.lane_stream[l]);
    }
  } drain{cx};
  for (int b = 0; b < nblk; ++b) {
    const int cb0 = (c1 - 1) + (int)(((long long)cN * b) / nblk), cb1 = (c1 - 1) + (int)(((long long)cN * (b + 1)) / nblk);
    if (cb1 <= cb0) continue;
    const size_t lb0 = (b == 0) ? l1 : layer_begin(cb0), lb1 = (b == nblk - 1) ? l2 : layer_begin(cb1);
    rc = sg.copy_window(true, (size_t)cb0, (size_t)cb1, lb0, lb1, s_up);
    if (rc) return rc;
    if (nblk > 1) {
      SSB_CUDA(cudaEventRecord(cx.blk_events[2 * b], s_up));
      SSB_CUDA(cudaStreamWaitEvent(s_run, cx.blk_events[2 * b], 0));
    }
    // input stage of the window: default contact fraction, emission from temperatures
    ds.derive(dcp, config->min_vegetation_fraction, (size_t)cb0, (size_t)cb1, lb0, lb1, s_run);
    rc = run_window(cx, ca, 1, cx.budget_doubles, cb0, cb1);
    if (rc) return rc;
    if (drv) {  // scale + sum of the window (driver:250-261), still on the kernel lane
      const long cnt = (long)std::max((size_t)(cb1 - cb0), lb1 - lb0);
      auto scale_sum = [&](ssb200_canopy_flux &o, ssb200_canopy_flux &x, ssb200_canopy_flux &y, const double *fa,
                           const double *fb, const double *fbm, int nspec) {
        FieldList fl;
        collect_fields(&o, &x, &y, fl, true);
        const long nthr = cnt * nspec;
        if (fl.n == 0 || nthr <= 0) return;
        k_scale_sum<double><<<(unsigned)((nthr + 255) / 256), 256, 0, s_run>>>(fl, fa, fb, fbm, (const int *)cx.d_lay2col.p, nspec,
                                                                       (long)cb0, (long)cb1, (long)lb0, (long)lb1);
        ++g_launches;
      };
      if (config->do_sw) scale_sum(dsum_sw, d1, d2, d_top_dir, d_top_sw, d_top_dir, config->nsw);
      if (config->do_lw) scale_sum(dsum_lw, d3, d4, nullptr, d_top_lw, nullptr, config->nlw);
      SSB_CUDA(cudaGetLastError());
    }
    if (nblk > 1) {
      SSB_CUDA(cudaEventRecord(cx.blk_events[2 * b + 1], s_run));
      SSB_CUDA(cudaStreamWaitEvent(s_down, cx.blk_events[2 * b + 1], 0));
    }
    rc = sg.copy_window(false, (size_t)cb0, (size_t)cb1, lb0, lb1, s_down);
    if (rc) return rc;
  }
  for (int l = 0; l < Context::kLanes; ++l) SSB_CUDA(cudaStreamSynchronize(cx.lane_stream[l]));
  drain.armed = false;
  int status = 0;
  SSB_CUDA(cudaMemcpy(&status, cx.d_status.p, sizeof(int), cudaMemcpyDeviceToHost));
  return status;
}

int ssb200_radsurf(const ssb200_config *config, const ssb200_canopy_properties *cp,
                   const ssb200_sw_spectral_properties *sw, const ssb200_lw_spectral_properties *lw,
                   ssb200_boundary_conds_out *bc, int32_t istartcol, int32_t iendcol, ssb200_canopy_flux *sw_dir,
                   ssb200_canopy_flux *sw_diff, ssb200_canopy_flux *lw_int, ssb200_canopy_flux *lw_norm) {
  return radsurf_host(config, cp, sw, lw, nullptr, bc, istartcol, iendcol, sw_dir, sw_diff, lw_int, lw_norm, nullptr,
                      nullptr);
}

int ssb200_radsurf_fluxes(const ssb200_config *config, const ssb200_canopy_properties *cp,
                          const ssb200_sw_spectral_properties *sw, const ssb200_lw_spectral_properties *lw,
                          const ssb200_driver_inputs *drv, ssb200_boundary_conds_out *bc, int32_t istartcol,
                          int32_t iendcol, ssb200_canopy_flux *sw_flux, ssb200_canopy_flux *lw_flux) {
  if (!drv) return fail(SSB200_ERR_ARG, "driver_inputs must not be NULL");
  return radsurf_host(config, cp, sw, lw, drv, bc, istartcol, iendcol, nullptr, nullptr, nullptr, nullptr, sw_flux,
                      lw_flux);
}

// Single-precision storage variant (-DSINGLE_PRECISION builds of the reference: jprb = real32,
// utilities/parkind1.F90:45-49).  The _sp structs are layout-identical to the double ones (pointers
// and 32-bit integers only), so the body is shared; the Stager widens / rounds on the device.
int ssb200_radsurf_sp(const ssb200_config *config, const ssb200_canopy_properties_sp *cp,
                      const ssb200_sw_spectral_properties_sp *sw, const ssb200_lw_spectral_properties_sp *lw,
                      ssb200_boundary_conds_out_sp *bc, int32_t istartcol, int32_t iendcol, ssb200_canopy_flux_sp *sw_dir,
                      ssb200_canopy_flux_sp *sw_diff, ssb200_canopy_flux_sp *lw_int, ssb200_canopy_flux_sp *lw_norm) {
  static_assert(sizeof(ssb200_canopy_properties_sp) == sizeof(ssb200_canopy_properties) &&
                    sizeof(ssb200_sw_spectral_properties_sp) == sizeof(ssb200_sw_spectral_properties) &&
                    sizeof(ssb200_lw_spectral_properties_sp) == sizeof(ssb200_lw_spectral_properties) &&
                    sizeof(ssb200_canopy_flux_sp) == sizeof(ssb200_canopy_flux) &&
                    sizeof(ssb200_boundary_conds_out_sp) == sizeof(ssb200_boundary_conds_out) &&
                    sizeof(ssb200_driver_inputs_sp) == sizeof(ssb200_driver_inputs),
                "single-precision structs must mirror the double-precision ones");
  return radsurf_host(config, reinterpret_cast<const ssb200_canopy_properties *>(cp),
                      reinterpret_cast<const ssb200_sw_spectral_properties *>(sw),
                      reinterpret_cast<const ssb200_lw_spectral_properties *>(lw), nullptr,
                      reinterpret_cast<ssb200_boundary_conds_out *>(bc), istartcol, iendcol,
                      reinterpret_cast<ssb200_canopy_flux *>(sw_dir), reinterpret_cast<ssb200_canopy_flux *>(sw_diff),
                      reinterpret_cast<ssb200_canopy_flux *>(lw_int), reinterpret_cast<ssb200_canopy_flux *>(lw_norm), nullptr,
                      nullptr, true);
}

int ssb200_radsurf_fluxes_sp(const ssb200_config *config, const ssb200_canopy_properties_sp *cp,
                             const ssb200_sw_spectral_properties_sp *sw, const ssb200_lw_spectral_properties_sp *lw,
                             const ssb200_driver_inputs_sp *drv, ssb200_boundary_conds_out_sp *bc, int32_t istartcol,
                             int32_t iendcol, ssb200_canopy_flux_sp *sw_flux, ssb200_canopy_flux_sp *lw_flux) {
  if (!drv) return fail(SSB200_ERR_ARG, "driver_inputs must not be NULL");
  return radsurf_host(config, reinterpret_cast<const ssb200_canopy_properties *>(cp),
                      reinterpret_cast<const ssb200_sw_spectral_properties *>(sw),
                      reinterpret_cast<const ssb200_lw_spectral_properties *>(lw),
                      reinterpret_cast<const ssb200_driver_inputs *>(drv), reinterpret_cast<ssb200_boundary_conds_out *>(bc),
                      istartcol, iendcol, nullptr, nullptr, nullptr, nullptr, reinterpret_cast<ssb200_canopy_flux *>(sw_flux),
                      reinterpret_cast<ssb200_canopy_flux *>(lw_flux), true);
}

int ssb200_radsurf_device_sp(const ssb200_config *config, const ssb200_canopy_properties_sp *cp,
                             const ssb200_sw_spectral_properties_sp *sw, const ssb200_lw_spectral_properties_sp *lw,
                             ssb200_boundary_conds_out_sp *bc, int32_t istartcol, int32_t iendcol,
                             ssb200_canopy_flux_sp *sw_norm_dir, ssb200_canopy_flux_sp *sw_norm_diff,
                             ssb200_canopy_flux_sp *lw_internal, ssb200_canopy_flux_sp *lw_norm, void *stream,
                             int32_t *status_out) {
  int rc = ensure_device();
  if (rc) return rc;
  std::lock_guard<std::mutex> lock(g_mutex);
  ssb::CallArgs ca{config,
                   reinterpret_cast<const ssb200_canopy_properties *>(cp),
                   reinterpret_cast<const ssb200_sw_spectral_properties *>(sw),
                   reinterpret_cast<const ssb200_lw_spectral_properties *>(lw),
                   reinterpret_cast<ssb200_boundary_conds_out *>(bc),
                   reinterpret_cast<ssb200_canopy_flux *>(sw_norm_dir),
                   reinterpret_cast<ssb200_canopy_flux *>(sw_norm_diff),
                   reinterpret_cast<ssb200_canopy_flux *>(lw_internal),
                   reinterpret_cast<ssb200_canopy_flux *>(lw_norm)};
  return radsurf_device_sp_locked(g_ctx, ca, istartcol, iendcol, (cudaStream_t)stream, status_out);
}

int ssb200_radsurf_fluxes_device(const ssb200_config *config, const ssb200_canopy_properties *canopy_props,
                                 const ssb200_sw_spectral_properties *sw, const ssb200_lw_spectral_properties *lw,
                                 const ssb200_driver_inputs *driver_inputs, ssb200_boundary_conds_out *bc_out,
                                 int32_t istartcol, int32_t iendcol, ssb200_canopy_flux *sw_flux,
                                 ssb200_canopy_flux *lw_flux, void *stream, int32_t *status_out) {
  int rc = ensure_device();
  if (rc) return rc;
  std::lock_guard<std::mutex> lock(g_mutex);
  return radsurf_fluxes_device_locked(g_ctx, config, canopy_props, sw, lw, driver_inputs, bc_out, istartcol, iendcol,
                                      sw_flux, lw_flux, (cudaStream_t)stream, status_out);
}

int ssb200_radsurf_fluxes_device_sp(const ssb200_config *config, const ssb200_canopy_properties_sp *canopy_props,
                                    const ssb200_sw_spectral_properties_sp *sw,
                                    const ssb200_lw_spectral_properties_sp *lw,
                                    const ssb200_driver_inputs_sp *driver_inputs, ssb200_boundary_conds_out_sp *bc_out,
                                    int32_t istartcol, int32_t iendcol, ssb200_canopy_flux_sp *sw_flux,
                                    ssb200_canopy_flux_sp *lw_flux, void *stream, int32_t *status_out) {
  int rc = ensure_device();
  if (rc) return rc;
  std::lock_guard<std::mutex> lock(g_mutex);
  return radsurf_fluxes_device_locked(g_ctx, config, reinterpret_cast<const ssb200_canopy_properties *>(canopy_props),
                                      reinterpret_cast<const ssb200_sw_spectral_properties *>(sw),
                                      reinterpret_cast<const ssb200_lw_spectral_properties *>(lw),
                                      reinterpret_cast<const ssb200_driver_inputs *>(driver_inputs),
                                      reinterpret_cast<ssb200_boundary_conds_out *>(bc_out), istartcol, iendcol,
                                      reinterpret_cast<ssb200_canopy_flux *>(sw_flux),
                                      reinterpret_cast<ssb200_canopy_flux *>(lw_flux), (cudaStream_t)stream, status_out,
                                      true);
}

int64_t ssb200_kernel_launch_count(void) { return (int64_t)g_launches; }

int ssb200_set_profiling(int enable) {
  std::lock_guard<std::mutex> lock(g_mutex);
  g_ctx.profiling = enable != 0;
  return 0;
}

int ssb200_last_kernel_times_ms(double out[5]) {
  std::lock_guard<std::mutex> lock(g_mutex);
  for (int i = 0; i < 5; ++i) out[i] = g_ctx.times_ms[i];
  return 0;
}

int ssb200_last_kernel_counts(int64_t out[5]) {
  std::lock_guard<std::mutex> lock(g_mutex);
  for (int i = 0; i < 5; ++i) out[i] = g_ctx.counts[i];
  return 0;
}

int ssb200_set_option(const char *name, int64_t value) {
  std::lock_guard<std::mutex> lock(g_mutex);
  const std::string n(name ? name : "");
  if (n == "scratch_budget_bytes") {
    g_ctx.budget_doubles = (size_t)value / sizeof(double);
    return 0;
  }
  if (n == "fast_kernels") {
    g_ctx.fast_mode = value != 0;
    return 0;
  }
  if (n == "pipeline") {
    g_ctx.pipeline = value != 0;
    return 0;
  }
  if (n == "sort_columns") {
    g_ctx.sort_columns = value != 0;
    return 0;
  }
  if (n == "sort_group") {
    g_ctx.sort_group = (int)value;
    return 0;
  }
  if (n == "pipeline_max_blocks") {
    g_ctx.pipeline_max_blocks = value < 1 ? 1 : (int)value;
    return 0;
  }
  if (n == "concurrent_passes") {
    g_ctx.concurrent_passes = value != 0;
    return 0;
  }
  if (n == "stage_layers") {
    g_ctx.stage_layers = value != 0;
    return 0;
  }
  if (n == "record_sweeps") {
    g_ctx.sweep_mode = value != 0 ? 1 : 0;
    return 0;
  }
  if (n == "fused_kernels") {  // column-resident kernels where they exist (1 and 2 streams)
    g_ctx.fused_mode = value != 0;
    return 0;
  }
  if (n == "fused_sort") {
    g_ctx.fused_sort = value != 0;
    return 0;
  }
  if (n == "fused_sort_group") {
    g_ctx.fused_sort_group = (int)value;
    return 0;
  }
  if (n == "fused_blocks_per_sm") {
    g_ctx.fused_blocks_per_sm = value < 1 ? 1 : (value > 2 ? 2 : (int)value);
    return 0;
  }
  if (n == "fused_sync") {
    g_ctx.fused_sync = value != 0;
    return 0;
  }
  if (n == "fused_l2_persist") {
    g_ctx.fused_l2_persist = value != 0;
    return 0;
  }
  if (n == "partition_layers") {
    g_ctx.partition = value != 0;
    return 0;
  }
  return fail(SSB200_ERR_ARG, "unknown option " + n);
}

int ssb200_release(void) {
  std::lock_guard<std::mutex> lock(g_mutex);
  Context &cx = g_ctx;
  if (ssb200_device_count() > 0) {
    cudaDeviceSynchronize();
    for (DevBuf *b : {&cx.d_nlay, &cx.d_istart, &cx.d_irep, &cx.d_cols, &cx.d_status, &cx.d_lay2col}) b->release();
    for (int l = 0; l < Context::kLanes; ++l) {
      cx.d_scratch[l].release();
      cx.d_perm[l].release();
      cx.d_sort[l].release();
    }
    for (DevBuf &b : cx.stage) b.release();
    for (DevBuf &b : cx.wide) b.release();
    for (DevBuf &b : cx.drv) b.release();
  }
  cx.plan = ssb::Plan();
  cx.plan_uploaded = false;
  cx.budget_doubles = 0;
  return 0;
}

int ssb200_canopy_flux_scale_device(ssb200_canopy_flux *flux, const int32_t *nlay, const int32_t *istartlay,
                                    const double *factor, void *stream) {
  int rc = ensure_device();
  if (rc) return rc;
  if (!flux || !nlay || !istartlay || !factor) return fail(SSB200_ERR_ARG, "NULL argument");
  std::lock_guard<std::mutex> lock(g_mutex);
  Context &cx = g_ctx;
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<int> lay2col((size_t)flux->ntotlay, 0);
  for (int j = 0; j < flux->ncol; ++j)
    for (int l = 0; l < nlay[j]; ++l) {
      const long il = (long)istartlay[j] - 1 + l;
      if (il < 0 || il >= flux->ntotlay) return fail(SSB200_ERR_SHAPE, "layer range outside 1..ntotlay");
      lay2col[(size_t)il] = j;
    }
  SSB_CUDA(cx.d_lay2col.reserve(sizeof(int) * (lay2col.size() + 1)));
  cx.lay2col_generation = -1;  // (the plan's map is rebuilt by the next call that needs it)
  SSB_CUDA(cudaMemcpyAsync(cx.d_lay2col.p, lay2col.data(), sizeof(int) * lay2col.size(), cudaMemcpyHostToDevice, st));
  SSB_CUDA(cudaStreamSynchronize(st));
  FieldList fl;
  collect_fields(flux, nullptr, nullptr, fl, false);
  const long nmax = (long)(flux->ntotlay > flux->ncol ? flux->ntotlay : flux->ncol) * flux->nspec;
  if (nmax > 0) {
    k_scale<<<(unsigned)((nmax + 255) / 256), 256, 0, st>>>(fl, factor, (const int *)cx.d_lay2col.p, flux->nspec,
                                                            flux->ncol, flux->ntotlay);
    ++g_launches;
    SSB_CUDA(cudaGetLastError());
  }
  return 0;
}

int ssb200_canopy_flux_sum_device(ssb200_canopy_flux *out, const ssb200_canopy_flux *a, const ssb200_canopy_flux *b,
                                  void *stream) {
  int rc = ensure_device();
  if (rc) return rc;
  if (!out || !a || !b) return fail(SSB200_ERR_ARG, "NULL argument");
  FieldList fl;
  collect_fields(out, a, b, fl, true);
  const long nmax = (long)(out->ntotlay > out->ncol ? out->ntotlay : out->ncol) * out->nspec;
  if (nmax > 0) {
    k_sum<<<(unsigned)((nmax + 255) / 256), 256, 0, (cudaStream_t)stream>>>(fl, out->nspec, out->ncol, out->ntotlay);
    ++g_launches;
    SSB_CUDA(cudaGetLastError());
  }
  return 0;
}

int ssb200_canopy_flux_check_device(const ssb200_canopy_flux *flux, const ssb200_canopy_properties *cp,
                                    double *residual, void *stream) {
  int rc = ensure_device();
  if (rc) return rc;
  if (!flux || !cp || !residual) return fail(SSB200_ERR_ARG, "NULL argument");
  std::lock_guard<std::mutex> lock(g_mutex);
  Context &cx = g_ctx;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t ncol = (size_t)cp->ncol;
  SSB_CUDA(cx.d_nlay.reserve(sizeof(int) * (ncol + 1)));
  SSB_CUDA(cx.d_istart.reserve(sizeof(int) * (ncol + 1)));
  SSB_CUDA(cx.d_irep.reserve(sizeof(int) * (ncol + 1)));
  SSB_CUDA(cudaMemcpyAsync(cx.d_nlay.p, cp->nlay, sizeof(int) * ncol, cudaMemcpyHostToDevice, st));
  SSB_CUDA(cudaMemcpyAsync(cx.d_istart.p, cp->istartlay, sizeof(int) * ncol, cudaMemcpyHostToDevice, st));
  SSB_CUDA(cudaMemcpyAsync(cx.d_irep.p, cp->i_representation, sizeof(int) * ncol, cudaMemcpyHostToDevice, st));
  SSB_CUDA(cudaStreamSynchronize(st));
  cx.plan_uploaded = false;  // the index buffers were overwritten
  cx.plan.valid = false;
  if (ncol > 0) {
    k_check<<<(unsigned)((ncol + 127) / 128), 128, 0, st>>>(*flux, (const int *)cx.d_nlay.p, (const int *)cx.d_istart.p,
                                                            (const int *)cx.d_irep.p, (int)ncol, residual);
    ++g_launches;
    SSB_CUDA(cudaGetLastError());
  }
  return 0;
}

int ssb200_calc_simple_spectrum_lw_device(ssb200_lw_spectral_properties *lw, int32_t ncol, int32_t ntotlay,
                                          int32_t istartcol, int32_t iendcol, int32_t ilay1, int32_t ilay2,
                                          const double *ground_temperature, const double *roof_temperature,
                                          const double *wall_temperature, const double *clear_air_temperature,
                                          const double *veg_temperature, const double *veg_air_temperature,
                                          void *stream) {
  int rc = ensure_device();
  if (rc) return rc;
  if (!lw) return fail(SSB200_ERR_ARG, "NULL argument");
  if (lw->nspec > 1 && (clear_air_temperature || veg_temperature || veg_air_temperature))
    return fail(SSB200_ERR_ARG, "Simple longwave spectrum only possible with one input spectral interval");
  const long c0 = (istartcol > 0 ? istartcol : 1) - 1, c1 = iendcol > 0 ? (iendcol < ncol ? iendcol : ncol) : ncol;
  const long l0 = (ilay1 > 0 ? ilay1 : 1) - 1, l1 = ilay2 < ntotlay ? ilay2 : ntotlay;
  cudaStream_t st = (cudaStream_t)stream;
  // (the members are inputs of radsurf, hence const in the struct; this stage fills them)
  auto run = [&](const double *out_c, const double *emis, const double *temp, long i0, long i1, bool need_emis) -> int {
    double *out = const_cast<double *>(out_c);
    if (!temp || i1 <= i0) return 0;
    if (!out || (need_emis && !emis)) return fail(SSB200_ERR_ARG, "temperature given but emission / emissivity array missing");
    k_sigma_t4<double><<<(unsigned)((i1 - i0 + 255) / 256), 256, 0, st>>>(out, emis, temp, lw->nspec, i0, i1);
    ++g_launches;
    SSB_CUDA(cudaGetLastError());
    return 0;
  };
  if ((rc = run(lw->ground_emission, lw->ground_emissivity, ground_temperature, c0, c1, true))) return rc;
  if ((rc = run(lw->roof_emission, lw->roof_emissivity, roof_temperature, l0, l1, true))) return rc;
  if ((rc = run(lw->wall_emission, lw->wall_emissivity, wall_temperature, l0, l1, true))) return rc;
  if ((rc = run(lw->clear_air_planck, nullptr, clear_air_temperature, l0, l1, false))) return rc;
  if ((rc = run(lw->veg_planck, nullptr, veg_temperature, l0, l1, false))) return rc;
  if ((rc = run(lw->veg_air_planck, nullptr, veg_air_temperature, l0, l1, false))) return rc;
  return 0;
}

double ssb200_measure_fp64_peak_tflops(int iters) {
  if (ensure_device()) return -1.0;
  if (iters <= 0) iters = 1 << 16;
  cudaDeviceProp prop;
  int dev = 0;
  cudaGetDevice(&dev);
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return -1.0;
  const int blocks = prop.multiProcessorCount * 8, threads = 256;
  double *out = nullptr;
  if (cudaMalloc(&out, sizeof(double) * blocks * threads) != cudaSuccess) return -1.0;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(e0);
    k_fp64_peak<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    const double tf = 2.0 * 8.0 * (double)iters * blocks * threads / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  ++g_launches;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  if (cudaGetLastError() != cudaSuccess) return -1.0;
  return best;
}

}  // extern "C"
