// ssb_stage.cuh - level-major staging of the per-layer arrays of one chunk of columns.
//
// The reference layout packs the layers of a column contiguously ((nspec, ntotlay) arrays, layer
// il = istartlay(col) - 1 + lev).  The register-resident kernels run one thread per column (or per
// column and level), so in that layout the threads of a warp touch addresses nlay * nspec doubles
// apart: every 8-byte access moves its own 32-byte sector, and with ~40 k threads in flight the
// partially used sectors do not survive in L2 until their neighbours are touched (ncu, round 2:
// 3.1 KB of DRAM traffic per (column, layer) in a kernel whose useful bytes are 0.9 KB).  The C-ABI
// therefore does what the north-star describes for the shim: it repacks the per-layer inputs of a
// chunk into structure-of-arrays buffers ordered [level][column][interval] ("gather"), lets the
// kernels read and write those with consecutive addresses per warp, and copies the per-layer outputs
// back into the caller's arrays ("scatter").  Both directions go through a shared-memory tile so
// that reads and writes are full sectors on both sides.
#pragma once
#include "ssb_solver.cuh"

namespace ssb {

constexpr int kStageMaxArrays = 40;
struct StageList {
  int n;
  double *ref[kStageMaxArrays];     // the caller's array, reference layout (inputs are not written)
  double *staged[kStageMaxArrays];  // [lev][ic][g] buffer of the chunk
  int nspec[kStageMaxArrays];
  // 1: `ref` really holds float (ssb200_radsurf_device_sp, ssb200_radsurf_fluxes_device_sp): the gather
  // widens exactly, the scatter rounds to nearest, so the kernels see the same doubles as the double entry
  // on widened inputs.  Set per array: one list may mix the caller's float arrays with double buffers.
  unsigned char f32[kStageMaxArrays];
  // summing scatter (ssb200_radsurf_fluxes_device and _sp): `ref` is a member of the summed flux object and
  // receives a combination of `staged` (the member of f1) and `staged2` (the same member of f2), summed in
  // FP64 and, when f32 is set, rounded once to float.
  // kSumScaled: fa * a + (fb - fb_minus) * b per (interval, column); kSumPlain: a + b (sunlit fractions)
  unsigned char sum[kStageMaxArrays];
  double *staged2[kStageMaxArrays];
};
enum { kSumNone = 0, kSumScaled = 1, kSumPlain = 2 };
struct StageArgs {
  StageList list;
  const int *cols, *nlay, *istartlay;
  int ncols, lmax;
  // factors of the summing scatter, (nspec, ncol) in reference layout: fa NULL means 1, fb_minus
  // non-NULL means fb - fb_minus (canopy_flux_type%scale followed by %sum, driver:250-261)
  const double *fa, *fb, *fb_minus;
};

// One summed value, rounded as canopy_flux_type%scale (one product per object) followed by %sum
// (radsurf/radsurf_canopy_flux.F90:212-282,399-460); `f` indexes the factors, g + nspec * col.
// Written with explicit round-to-nearest operations so that no FMA contraction changes the bits.
SSB_HDI double stage_sum(const StageArgs &s, int k, double a, double b, size_t f) {
#if defined(__CUDA_ARCH__)
  if (s.list.sum[k] == kSumPlain) return __dadd_rn(a, b);
  const double xa = s.fa ? __dmul_rn(s.fa[f], a) : a;
  const double fbk = s.fb_minus ? __dadd_rn(s.fb[f], -s.fb_minus[f]) : s.fb[f];
  return __dadd_rn(xa, __dmul_rn(fbk, b));
#else  // (the host check is compiled with -ffp-contract=off)
  if (s.list.sum[k] == kSumPlain) return a + b;
  const double xa = s.fa ? s.fa[f] * a : a;
  const double fbk = s.fb_minus ? s.fb[f] - s.fb_minus[f] : s.fb[f];
  return xa + fbk * b;
#endif
}

// serial form (host check)
inline void stage_host(const StageArgs &s, bool scatter) {
  for (int k = 0; k < s.list.n; ++k) {
    const int ns = s.list.nspec[k];
    for (int ic = 0; ic < s.ncols; ++ic) {
      const int col = s.cols[ic], il1 = s.istartlay[col] - 1;
      for (int lev = 0; lev < s.nlay[col]; ++lev)
        for (int g = 0; g < ns; ++g) {
          const size_t ri = (size_t)g + (size_t)ns * (size_t)(il1 + lev);
          const size_t si = (size_t)g + (size_t)ns * ((size_t)ic + (size_t)lev * (size_t)s.ncols);
          double &t = s.list.staged[k][si];
          if (s.list.sum[k]) {  // (scatter only)
            const double v = stage_sum(s, k, t, s.list.staged2[k][si], (size_t)g + (size_t)ns * (size_t)col);
            if (s.list.f32[k])
              reinterpret_cast<float *>(s.list.ref[k])[ri] = (float)v;  // round to nearest even
            else
              s.list.ref[k][ri] = v;
          } else if (s.list.f32[k]) {
            float &r = reinterpret_cast<float *>(s.list.ref[k])[ri];
            if (scatter)
              r = (float)t;  // round to nearest even
            else
              t = (double)r;
          } else {
            double &r = s.list.ref[k][ri];
            if (scatter)
              r = t;
            else
              t = r;
          }
        }
    }
  }
}

#if defined(__CUDACC__)
constexpr int kStageBlock = 256;
constexpr int kStageTile = 4096;  // doubles of shared memory per block
// store of a staged double on the caller's side: unchanged, or rounded to nearest float
__device__ __forceinline__ double stage_out(double *, double v) { return v; }
__device__ __forceinline__ float stage_out(float *, double v) { return __double2float_rn(v); }

// blockIdx.x: tile of `tc` chunk columns, blockIdx.y: array.  `lb` levels per pass of the tile.
// R: element type of the caller's side (double, or float for the single-precision device entry).
// SUM: summing scatter (StageList::sum): the tile receives the combination of both staged objects.
template <bool SCATTER, class R, bool SUM = false>
__global__ void __launch_bounds__(kStageBlock) k_stage(StageArgs s, int tc, int lb) {
  __shared__ double tile[kStageTile + 2 * 64];
  const int k = blockIdx.y, ns = s.list.nspec[k];
  R *ref = reinterpret_cast<R *>(s.list.ref[k]);
  double *stg = s.list.staged[k];
  const int ic0 = blockIdx.x * tc;
  const int ncl = min(tc, s.ncols - ic0);
  if (ncl <= 0) return;
  const int row = ncl * ns, pitch = row | 1;  // odd pitch: the two access patterns stay conflict-poor
  for (int l0 = 0; l0 < s.lmax; l0 += lb) {
    const int nl = min(lb, s.lmax - l0);
    const int total = row * nl;
    if (!SCATTER) {
      for (int idx = threadIdx.x; idx < total; idx += kStageBlock) {  // (l, g) fastest: contiguous in `ref`
        const int c = idx / (nl * ns), r = idx % (nl * ns), l = r / ns, g = r % ns;
        const int col = s.cols[ic0 + c];
        if (l0 + l < s.nlay[col])
          tile[l * pitch + c * ns + g] = (double)ref[(size_t)g + (size_t)ns * (size_t)(s.istartlay[col] - 1 + l0 + l)];
      }
      __syncthreads();
      for (int idx = threadIdx.x; idx < total; idx += kStageBlock) {  // (c, g) fastest: contiguous in `stg`
        const int l = idx / row, r = idx % row, c = r / ns;
        if (l0 + l < s.nlay[s.cols[ic0 + c]])
          stg[(size_t)(r % ns) + (size_t)ns * ((size_t)(ic0 + c) + (size_t)(l0 + l) * (size_t)s.ncols)] = tile[l * pitch + r];
      }
    } else {
      for (int idx = threadIdx.x; idx < total; idx += kStageBlock) {
        const int l = idx / row, r = idx % row, c = r / ns;
        const int col = s.cols[ic0 + c];
        if (l0 + l < s.nlay[col]) {
          const size_t si = (size_t)(r % ns) + (size_t)ns * ((size_t)(ic0 + c) + (size_t)(l0 + l) * (size_t)s.ncols);
          if constexpr (SUM)
            tile[l * pitch + r] = stage_sum(s, k, stg[si], s.list.staged2[k][si], (size_t)(r % ns) + (size_t)ns * (size_t)col);
          else
            tile[l * pitch + r] = stg[si];
        }
      }
      __syncthreads();
      for (int idx = threadIdx.x; idx < total; idx += kStageBlock) {
        const int c = idx / (nl * ns), r = idx % (nl * ns), l = r / ns, g = r % ns;
        const int col = s.cols[ic0 + c];
        if (l0 + l < s.nlay[col])
          ref[(size_t)g + (size_t)ns * (size_t)(s.istartlay[col] - 1 + l0 + l)] = stage_out(ref, tile[l * pitch + c * ns + g]);
      }
    }
    __syncthreads();
  }
}

// Arrays with one value per layer (every array when nsw = nlw = 1): no tile needed.  A thread moves four
// vertically adjacent layers of one column of every array: on the reference side that is one full 32-byte
// sector per array (16 bytes for float), on the staged side four rows in which neighbouring threads are
// neighbouring columns.  SUM: summing scatter, as in k_stage.
template <bool SCATTER, class R, bool SUM = false>
__global__ void __launch_bounds__(kStageBlock) k_stage1(StageArgs s) {
  // neighbouring threads take neighbouring groups of four layers of ONE column: on the reference side a
  // warp then covers whole 128-byte lines (8 columns x 16 layers when every column has 16 layers)
  const long t = blockIdx.x * (long)kStageBlock + threadIdx.x;
  const int ng = (s.lmax + 3) / 4;
  const int ic = (int)(t / ng), l0 = 4 * (int)(t % ng);
  if (ic >= s.ncols) return;
  const int col = s.cols[ic];
  const int cnt = s.nlay[col] - l0;
  if (cnt <= 0) return;
  const size_t rbase = (size_t)(s.istartlay[col] - 1 + l0);
  const size_t sbase = (size_t)ic + (size_t)l0 * (size_t)s.ncols;
  const size_t pitch = (size_t)s.ncols;
  const bool vec = cnt >= 4 && (rbase & 1) == 0;  // two aligned 16-byte accesses on the reference side
#pragma unroll 4
  for (int k = 0; k < s.list.n; ++k) {
    R *ref = reinterpret_cast<R *>(s.list.ref[k]) + rbase;
    double *stg = s.list.staged[k] + sbase;
    double v[4];
    if constexpr (sizeof(R) == sizeof(float)) {
      // four floats are one 16-byte access when the ADDRESS is 16-byte aligned (the caller's base
      // address is not assumed to be)
      const bool vec4 = cnt >= 4 && ((size_t)ref & 15) == 0;
      if (!SCATTER) {
        if (vec4) {
          const float4 a = __ldcs((const float4 *)ref);
          v[0] = a.x, v[1] = a.y, v[2] = a.z, v[3] = a.w;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < cnt) v[j] = (double)__ldcs(ref + j);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < cnt) stg[j * pitch] = v[j];
      } else {
        if constexpr (SUM) {  // summed in FP64, then rounded once
          const double *stg2 = s.list.staged2[k] + sbase;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < cnt) v[j] = stage_sum(s, k, __ldcs(stg + j * pitch), __ldcs(stg2 + j * pitch), (size_t)col);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < cnt) v[j] = __ldcs(stg + j * pitch);
        }
        if (vec4) {
          __stcs((float4 *)ref, make_float4(__double2float_rn(v[0]), __double2float_rn(v[1]), __double2float_rn(v[2]),
                                            __double2float_rn(v[3])));
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < cnt) __stcs(ref + j, __double2float_rn(v[j]));
        }
      }
    } else {
      if (!SCATTER) {
        if (vec) {
          const double2 a = __ldcs((const double2 *)ref), b = __ldcs((const double2 *)ref + 1);
          v[0] = a.x, v[1] = a.y, v[2] = b.x, v[3] = b.y;
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < cnt) v[j] = __ldcs(ref + j);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < cnt) stg[j * pitch] = v[j];
      } else {
        if constexpr (SUM) {
          const double *stg2 = s.list.staged2[k] + sbase;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < cnt) v[j] = stage_sum(s, k, __ldcs(stg + j * pitch), __ldcs(stg2 + j * pitch), (size_t)col);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < cnt) v[j] = __ldcs(stg + j * pitch);
        }
        if (vec) {
          __stcs((double2 *)ref, make_double2(v[0], v[1]));
          __stcs((double2 *)ref + 1, make_double2(v[2], v[3]));
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (j < cnt) __stcs(ref + j, v[j]);
        }
      }
    }
  }
}

template <bool SCATTER, class R, bool SUM = false>
inline void stage_launch_group(const StageArgs &g, int ns, cudaStream_t st) {
  if (ns == 1) {
    const long nthreads = (long)g.ncols * ((g.lmax + 3) / 4);
    const unsigned blocks = (unsigned)((nthreads + kStageBlock - 1) / kStageBlock);
    k_stage1<SCATTER, R, SUM><<<blocks, kStageBlock, 0, st>>>(g);
    return;
  }
  int lb = g.lmax < 32 ? g.lmax : 32;
  while (lb > 1 && lb * ns > kStageTile) lb /= 2;  // (stage_supported caps the spectral width at kStageTile)
  int tc = kStageTile / (lb * ns);
  tc = tc > 64 ? 64 : (tc < 1 ? 1 : tc);
  const dim3 grid((unsigned)((g.ncols + tc - 1) / tc), (unsigned)g.list.n);
  k_stage<SCATTER, R, SUM><<<grid, kStageBlock, 0, st>>>(g, tc, lb);
}

// launches one grid per group of arrays with the same spectral width (the tile shape depends on it) and
// the same element type on the caller's side (a summing scatter sums every array of its list: its
// scaled and plain members share the grid of their width)
inline void stage_launch(const StageArgs &s, bool scatter, cudaStream_t st, long *launches) {
  if (s.list.n == 0 || s.ncols <= 0 || s.lmax <= 0) return;
  int done[kStageMaxArrays] = {0};
  for (int k0 = 0; k0 < s.list.n; ++k0) {
    if (done[k0]) continue;
    StageArgs g = s;
    g.list.n = 0;
    const int ns = s.list.nspec[k0];
    const unsigned char f32 = s.list.f32[k0];
    const bool sum = s.list.sum[k0] != kSumNone;
    for (int k = k0; k < s.list.n; ++k)
      if (!done[k] && s.list.nspec[k] == ns && s.list.f32[k] == f32 && (s.list.sum[k] != kSumNone) == sum) {
        g.list.ref[g.list.n] = s.list.ref[k];
        g.list.staged[g.list.n] = s.list.staged[k];
        g.list.staged2[g.list.n] = s.list.staged2[k];
        g.list.nspec[g.list.n] = ns;
        g.list.f32[g.list.n] = f32;
        g.list.sum[g.list.n] = s.list.sum[k];
        ++g.list.n;
        done[k] = 1;
      }
    if (sum)  // (ssb200_radsurf_fluxes_device / _sp: the summed object's precision)
      f32 ? stage_launch_group<true, float, true>(g, ns, st) : stage_launch_group<true, double, true>(g, ns, st);
    else if (f32)
      scatter ? stage_launch_group<true, float>(g, ns, st) : stage_launch_group<false, float>(g, ns, st);
    else
      scatter ? stage_launch_group<true, double>(g, ns, st) : stage_launch_group<false, double>(g, ns, st);
    if (launches) ++*launches;
  }
}
#endif

}  // namespace ssb
