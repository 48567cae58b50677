// Linear resampling between physical image grids: ITK 5.1's ResampleImageFilter with an IdentityTransform and a
// LinearInterpolateImageFunction on float pixels, the first step of the reference's data pipeline (ResampleT1T2d,
// code/GAN/transforms.py:79-213: native scan -> the generator's 128^3 2 mm grid).  The arithmetic is the one pinned in
// include/mpgan.h, in fp64 with explicitly rounded operations (no contraction into FMA), so the result is bit-identical
// to the numpy restatement in oracle/resample.py.  Bit-parity with ITK itself is not claimed: ITK forms the continuous
// index incrementally along a row and inverts its matrix with vnl, which can differ in the last fp64 bits.
//
// One launch resamples `items` images of one geometry.  A warp owns 32 * kVox voxels of one output row; each thread
// takes kVox of them, 32 apart along x, so every store instruction of the warp is coalesced.  A thread first forms the
// continuous indices of all its voxels, then issues the (up to) 8 * kVox neighbour loads together, then lerps: the loads
// of a thread do not depend on one another.  A neighbour whose weight is 0 is replaced by the base voxel's address,
// so its value is never read (a NaN beside a grid-aligned sample cannot leak into it) and no load is predicated.
// Rank 2 is rank 3 with a trivial z; its kernel instance drops the z terms, which add exact zeros.
#include "common.cuh"

namespace mpgan {
namespace resample {

constexpr int kVox = 4;      // output voxels per thread
constexpr int kRows = 4;     // output rows per 128-thread block (one per warp)
constexpr int kMaxExtent = 1 << 22;

struct Map {
  double oo[3], m[9], oi[3], n[9];   // o_out, M_out (row-major), o_in, N_in (row-major); ITK axis order x, y, z
};

struct Ext {
  int in[3], out[3];                 // ITK axis order x, y, z
};

__device__ __forceinline__ double lerp(double a, double b, double d) {
  return __dadd_rn(a, __dmul_rn(__dsub_rn(b, a), d));
}

// One output row of the linear kernels; row = (item * out_z + iz) * out_y + iy.
template <bool kVol>
__device__ __forceinline__ void linear_row(const float* __restrict__ in, const Map& m, const Ext& e, int row, float dflt,
                                           float* __restrict__ out) {
  const int iy = row % e.out[1];
  const int rz = row / e.out[1];
  const int iz = kVol ? rz % e.out[2] : 0;
  const int64_t item = kVol ? rz / e.out[2] : rz;
  const int64_t plane = (int64_t)e.in[0] * e.in[1];
  const float* src = in + item * plane * e.in[2];
  const int xb = blockIdx.y * (32 * kVox) + threadIdx.x;
  const double fy = (double)iy, fz = (double)iz;

  int64_t off[kVox];
  int sx[kVox], sy[kVox];
  int64_t sz[kVox];
  double dx[kVox], dy[kVox], dz[kVox];
  bool inside[kVox];
#pragma unroll
  for (int v = 0; v < kVox; ++v) {
    const double fx = (double)(xb + 32 * v);
    double p[3], q[3], c[3];
#pragma unroll
    for (int k = 0; k < (kVol ? 3 : 2); ++k) {   // TransformIndexToPhysicalPoint
      p[k] = __dadd_rn(__dadd_rn(m.oo[k], __dmul_rn(m.m[3 * k], fx)), __dmul_rn(m.m[3 * k + 1], fy));
      if (kVol) p[k] = __dadd_rn(p[k], __dmul_rn(m.m[3 * k + 2], fz));
      q[k] = __dsub_rn(p[k], m.oi[k]);
    }
#pragma unroll
    for (int k = 0; k < (kVol ? 3 : 2); ++k) {   // TransformPhysicalPointToContinuousIndex
      c[k] = __dadd_rn(__dmul_rn(m.n[3 * k], q[0]), __dmul_rn(m.n[3 * k + 1], q[1]));
      if (kVol) c[k] = __dadd_rn(c[k], __dmul_rn(m.n[3 * k + 2], q[2]));
    }
    if (!kVol) c[2] = 0.0;
    bool ok = true;
    int b[3], s[3];
    double d[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      ok = ok && c[k] >= -0.5 && c[k] < (double)e.in[k] - 0.5;   // half-open; NaN fails both
      const double f = ok ? fmax(floor(c[k]), 0.0) : 0.0;
      const double dd = ok ? __dsub_rn(c[k], f) : 0.0;
      b[k] = (int)f;
      d[k] = dd > 0.0 ? dd : 0.0;
      s[k] = d[k] > 0.0 && b[k] + 1 < e.in[k] ? 1 : 0;   // upper neighbour min(b + 1, n - 1); none at weight 0
    }
    inside[v] = ok;
    off[v] = ok ? ((int64_t)b[2] * e.in[1] + b[1]) * e.in[0] + b[0] : 0;
    sx[v] = s[0];
    sy[v] = s[1] * e.in[0];
    sz[v] = s[2] * plane;
    dx[v] = d[0];
    dy[v] = d[1];
    dz[v] = d[2];
  }

  float a[kVox][8];
#pragma unroll
  for (int v = 0; v < kVox; ++v) {
    const float* p0 = src + off[v];
    a[v][0] = __ldg(p0);
    a[v][1] = __ldg(p0 + sx[v]);
    a[v][2] = __ldg(p0 + sy[v]);
    a[v][3] = __ldg(p0 + sy[v] + sx[v]);
    if (kVol) {
      const float* p1 = p0 + sz[v];
      a[v][4] = __ldg(p1);
      a[v][5] = __ldg(p1 + sx[v]);
      a[v][6] = __ldg(p1 + sy[v]);
      a[v][7] = __ldg(p1 + sy[v] + sx[v]);
    }
  }

  float* dst = out + (int64_t)row * e.out[0];
#pragma unroll
  for (int v = 0; v < kVox; ++v) {
    const int x = xb + 32 * v;
    if (x >= e.out[0]) break;
    // EvaluateOptimized's nesting: along x, then y, then z; a zero weight returns the lower value untouched
    const bool ux = dx[v] > 0.0, uy = dy[v] > 0.0;
    const double v00 = ux ? lerp(a[v][0], a[v][1], dx[v]) : (double)a[v][0];
    const double v01 = ux ? lerp(a[v][2], a[v][3], dx[v]) : (double)a[v][2];
    double r = uy ? lerp(v00, v01, dy[v]) : v00;
    if (kVol && dz[v] > 0.0) {
      const double v10 = ux ? lerp(a[v][4], a[v][5], dx[v]) : (double)a[v][4];
      const double v11 = ux ? lerp(a[v][6], a[v][7], dx[v]) : (double)a[v][6];
      r = lerp(r, uy ? lerp(v10, v11, dy[v]) : v10, dz[v]);
    }
    dst[x] = inside[v] ? __double2float_rn(r) : dflt;
  }
}

template <bool kVol>
__global__ void __launch_bounds__(128) resample_linear_kernel(const float* __restrict__ in, Map m, Ext e, int rows,
                                                              float dflt, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int row = blockIdx.x * kRows + threadIdx.y;
  if (row >= rows) return;
  linear_row<kVol>(in, m, e, row, dflt, out);
}

// Per-item maps in device memory (items x 24 fp64, the layout of map[24]): each warp stages its row's map in shared
// memory, and the voxels are then formed by exactly the arithmetic above.
__device__ __forceinline__ const Map& stage_map(const double* __restrict__ maps, const Ext& e, int row, Map* slot) {
  const int64_t item = row / ((int64_t)e.out[1] * e.out[2]);
  if (threadIdx.x < 24) reinterpret_cast<double*>(slot)[threadIdx.x] = maps[item * 24 + threadIdx.x];
  __syncwarp();
  return *slot;
}

template <bool kVol>
__global__ void __launch_bounds__(128) resample_linear_maps_kernel(const float* __restrict__ in,
                                                                   const double* __restrict__ maps, Ext e, int rows,
                                                                   float dflt, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  __shared__ Map sm[kRows];
  const int row = blockIdx.x * kRows + threadIdx.y;
  if (row >= rows) return;
  linear_row<kVol>(in, stage_map(maps, e, row, &sm[threadIdx.y]), e, row, dflt, out);
}

}  // namespace resample
}  // namespace mpgan

using namespace mpgan;

extern "C" int mpgan_resample_linear(const float* in, int64_t items, int32_t rank, const int32_t in_size[3],
                                     const int32_t out_size[3], const double map[24], float default_value, float* out,
                                     void* stream) {
  using namespace mpgan::resample;
  MPGAN_REQUIRE(in && out && in_size && out_size && map, MPGAN_ERR_SHAPE, "resample_linear: null pointer");
  MPGAN_REQUIRE(items >= 1, MPGAN_ERR_SHAPE, "resample_linear: items %lld (at least 1)", (long long)items);
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "resample_linear: rank %d (2 or 3)", (int)rank);
  Ext e;
  for (int k = 0; k < 3; ++k) {
    e.in[k] = in_size[k];
    e.out[k] = out_size[k];
    MPGAN_REQUIRE(e.in[k] >= 1 && e.in[k] <= kMaxExtent && e.out[k] >= 1 && e.out[k] <= kMaxExtent, MPGAN_ERR_SHAPE,
                  "resample_linear: axis %c: input extent %d, output extent %d (each in [1, 2^22])", "xyz"[k], e.in[k],
                  e.out[k]);
  }
  for (int i = 0; i < 24; ++i)
    MPGAN_REQUIRE(isfinite(map[i]), MPGAN_ERR_SHAPE, "resample_linear: map[%d] = %g is not finite", i, map[i]);
  Map m;
  for (int i = 0; i < 3; ++i) {
    m.oo[i] = map[i];
    m.oi[i] = map[12 + i];
  }
  for (int i = 0; i < 9; ++i) {
    m.m[i] = map[3 + i];
    m.n[i] = map[15 + i];
  }
  if (rank == 2) {
    MPGAN_REQUIRE(e.in[2] == 1 && e.out[2] == 1, MPGAN_ERR_SHAPE, "resample_linear: rank 2 with z extents %d, %d (must be 1)",
                  e.in[2], e.out[2]);
    const double* mats[2] = {m.m, m.n};
    for (int t = 0; t < 2; ++t)
      MPGAN_REQUIRE(mats[t][2] == 0.0 && mats[t][5] == 0.0 && mats[t][6] == 0.0 && mats[t][7] == 0.0 && mats[t][8] == 1.0,
                    MPGAN_ERR_SHAPE, "resample_linear: rank 2 needs the z row and column of %s to be the identity's",
                    t ? "N_in" : "M_out");
    MPGAN_REQUIRE(m.oo[2] == 0.0 && m.oi[2] == 0.0, MPGAN_ERR_SHAPE,
                  "resample_linear: rank 2 needs z origins 0, got %g and %g", m.oo[2], m.oi[2]);
  }
  const int64_t row_len = (int64_t)e.out[1] * e.out[2];
  MPGAN_REQUIRE(items <= 0x7fffffffLL / row_len, MPGAN_ERR_SHAPE,
                "resample_linear: %lld items of %lld output rows each exceed 2^31 - 1 rows", (long long)items,
                (long long)row_len);
  MPGAN_REQUIRE((double)items * e.in[0] * e.in[1] * e.in[2] < 0x1p62 && (double)items * e.out[0] * row_len < 0x1p62,
                MPGAN_ERR_SHAPE, "resample_linear: tensor too large");
  const int rows = (int)(items * row_len);
  const dim3 grid((unsigned)ceil_div(rows, kRows), (unsigned)ceil_div(e.out[0], 32 * kVox));
  if (rank == 3)
    launch_k(resample_linear_kernel<true>, grid, dim3(32, kRows), 0, (cudaStream_t)stream, in, m, e, rows,
             default_value, out);
  else
    launch_k(resample_linear_kernel<false>, grid, dim3(32, kRows), 0, (cudaStream_t)stream, in, m, e, rows,
             default_value, out);
  MPGAN_CHECK_LAUNCH("resample_linear_kernel");
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// Nearest-neighbour and cubic B-spline resampling (ITK's NearestNeighborInterpolateImageFunction and, order 3,
// BSplineDecompositionImageFilter + BSplineInterpolateImageFunction inside the same ResampleImageFilter).  The
// continuous index and the inside test are the linear kernel's operations in the linear kernel's order, restated in
// cindex() below; resample_linear_kernel keeps its own copy so that its code generation is unchanged.
//
// Nearest: the linear kernel's layout (a warp per 128 voxels of an output row, 4 per thread, 32 apart), one load per
// voxel.  Coefficients: one fp64 recursion per line, kept sequential (a scan would change the bits).  Along x a warp
// owns 32 rows and stages 32-column chunks of them in shared memory with coalesced loads and stores; each lane carries
// its row's recursion across the chunks, forward and then back.  Along y and z a thread owns a line and adjacent threads
// take adjacent x, so every access is coalesced.  Evaluation: one output voxel per thread (a warp per 32 voxels of a
// row), 64 independent fp64 coefficient loads at rank 3 (16 at rank 2), mostly from L1 / L2.
namespace mpgan {
namespace resample {

constexpr int kChunk = 32;   // columns of an x-pass chunk
constexpr int kHorizon = 18; // ITK's causal-initialisation horizon at tolerance 1e-10: ceil(log 1e-10 / log |z|)

struct Spline {
  double z, gain, k, iz;     // pole sqrt(3) - 2, (1 - z)(1 - 1/z), z / (z z - 1), 1 / z
};

__device__ __forceinline__ Spline spline_constants() {
  Spline s;
  s.z = __dsub_rn(__dsqrt_rn(3.0), 2.0);
  s.iz = __ddiv_rn(1.0, s.z);
  s.gain = __dmul_rn(__dsub_rn(1.0, s.z), __dsub_rn(1.0, s.iz));
  s.k = __ddiv_rn(s.z, __dsub_rn(__dmul_rn(s.z, s.z), 1.0));
  return s;
}

template <bool kVol>
__device__ __forceinline__ bool cindex(const Map& m, const Ext& e, double fx, double fy, double fz, double c[3]) {
  double p[3], q[3];
#pragma unroll
  for (int k = 0; k < (kVol ? 3 : 2); ++k) {   // TransformIndexToPhysicalPoint
    p[k] = __dadd_rn(__dadd_rn(m.oo[k], __dmul_rn(m.m[3 * k], fx)), __dmul_rn(m.m[3 * k + 1], fy));
    if (kVol) p[k] = __dadd_rn(p[k], __dmul_rn(m.m[3 * k + 2], fz));
    q[k] = __dsub_rn(p[k], m.oi[k]);
  }
#pragma unroll
  for (int k = 0; k < (kVol ? 3 : 2); ++k) {   // TransformPhysicalPointToContinuousIndex
    c[k] = __dadd_rn(__dmul_rn(m.n[3 * k], q[0]), __dmul_rn(m.n[3 * k + 1], q[1]));
    if (kVol) c[k] = __dadd_rn(c[k], __dmul_rn(m.n[3 * k + 2], q[2]));
  }
  if (!kVol) c[2] = 0.0;
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 3; ++k) ok = ok && c[k] >= -0.5 && c[k] < (double)e.in[k] - 0.5;   // half-open; NaN fails
  return ok;
}

template <typename T, bool kVol>
__device__ __forceinline__ void nearest_row(const T* __restrict__ in, const Map& m, const Ext& e, int row, T dflt,
                                            T* __restrict__ out) {
  const int iy = row % e.out[1];
  const int rz = row / e.out[1];
  const int iz = kVol ? rz % e.out[2] : 0;
  const int64_t item = kVol ? rz / e.out[2] : rz;
  const T* src = in + item * ((int64_t)e.in[0] * e.in[1] * e.in[2]);
  const int xb = blockIdx.y * (32 * kVox) + threadIdx.x;
  T v[kVox];
#pragma unroll
  for (int j = 0; j < kVox; ++j) {
    double c[3];
    const bool ok = cindex<kVol>(m, e, (double)(xb + 32 * j), (double)iy, (double)iz, c);
    int64_t off = 0;
    if (ok) {
      int i[3];
#pragma unroll
      for (int k = 0; k < 3; ++k) i[k] = min((int)floor(__dadd_rn(c[k], 0.5)), e.in[k] - 1);
      off = ((int64_t)i[2] * e.in[1] + i[1]) * e.in[0] + i[0];
    }
    v[j] = ok ? src[off] : dflt;
  }
  T* dst = out + (int64_t)row * e.out[0];
#pragma unroll
  for (int j = 0; j < kVox; ++j) {
    const int x = xb + 32 * j;
    if (x < e.out[0]) dst[x] = v[j];
  }
}

template <typename T, bool kVol>
__global__ void __launch_bounds__(128) resample_nearest_kernel(const T* __restrict__ in, Map m, Ext e, int rows,
                                                               T dflt, T* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int row = blockIdx.x * kRows + threadIdx.y;
  if (row >= rows) return;
  nearest_row<T, kVol>(in, m, e, row, dflt, out);
}

template <typename T, bool kVol>
__global__ void __launch_bounds__(128) resample_nearest_maps_kernel(const T* __restrict__ in,
                                                                    const double* __restrict__ maps, Ext e, int rows,
                                                                    T dflt, T* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  __shared__ Map sm[kRows];
  const int row = blockIdx.x * kRows + threadIdx.y;
  if (row >= rows) return;
  nearest_row<T, kVol>(in, stage_map(maps, e, row, &sm[threadIdx.y]), e, row, dflt, out);
}

// Causal initial value of a line whose first min(n, 18) gain-scaled values (and, when n <= 18, all n) are c(0..).
template <typename Get>
__device__ __forceinline__ double causal_init(const Spline& s, int n, Get c) {
  if (n > kHorizon) {
    double sum = c(0), zn = s.z;
#pragma unroll
    for (int j = 1; j < kHorizon; ++j) {
      sum = __dadd_rn(sum, __dmul_rn(zn, c(j)));
      zn = __dmul_rn(zn, s.z);
    }
    return sum;
  }
  double zl = s.z;                               // z^(n-1)
  for (int j = 2; j < n; ++j) zl = __dmul_rn(zl, s.z);
  double sum = __dadd_rn(c(0), __dmul_rn(zl, c(n - 1)));
  double a = s.z, b = __dmul_rn(zl, __dmul_rn(zl, s.iz));
  for (int j = 1; j <= n - 2; ++j) {
    sum = __dadd_rn(sum, __dmul_rn(__dadd_rn(a, b), c(j)));
    a = __dmul_rn(a, s.z);
    b = __dmul_rn(b, s.iz);
  }
  return __ddiv_rn(sum, __dsub_rn(1.0, __dmul_rn(a, a)));
}

// Along x: a warp owns 32 rows (lane r recurses row r) and walks them in chunks of 32 columns staged in shared memory.
// The forward sweep writes causal coefficients to coef except for the last chunk, which stays staged for the backward
// sweep.  The row stride of 33 doubles keeps a lane's column walk free of bank conflicts.
__global__ void __launch_bounds__(128) bspline_x_kernel(const float* __restrict__ in, double* __restrict__ coef, int nx,
                                                        int rows) {
  pdl_wait();
  pdl_launch();
  const Spline s = spline_constants();
  __shared__ double stage[4][32][kChunk + 1];
  double(*t)[kChunk + 1] = stage[threadIdx.y];
  const int lane = threadIdx.x;
  const int row0 = (blockIdx.x * 4 + threadIdx.y) * 32;
  if (row0 >= rows) return;
  const int nr = min(32, rows - row0);
  const bool mine = lane < nr;
  const float* src = in + (int64_t)row0 * nx;
  double* dst = coef + (int64_t)row0 * nx;
  const int last = (nx - 1) / kChunk * kChunk;   // first column of the last chunk
  const bool filt = nx > 1;
  double prev = 0.0, prev2 = 0.0;                // causal c[n-1], c[n-2] of this lane's row
  for (int x0 = 0; x0 <= last; x0 += kChunk) {
    const int w = min(kChunk, nx - x0);
    for (int r = 0; r < nr; ++r)
      if (lane < w) {
        const double v = (double)src[(int64_t)r * nx + x0 + lane];
        t[r][lane] = filt ? __dmul_rn(v, s.gain) : v;
      }
    __syncwarp();
    if (mine && filt) {
      int j0 = 0;
      if (x0 == 0) {
        prev = causal_init(s, nx, [&](int j) { return t[lane][j]; });
        t[lane][0] = prev;
        j0 = 1;
      }
      for (int j = j0; j < w; ++j) {
        const double c = __dadd_rn(t[lane][j], __dmul_rn(s.z, prev));
        t[lane][j] = c;
        prev2 = prev;
        prev = c;
      }
    }
    __syncwarp();
    if (x0 != last || !filt)
      for (int r = 0; r < nr; ++r)
        if (lane < w) dst[(int64_t)r * nx + x0 + lane] = t[r][lane];
    __syncwarp();
  }
  if (!filt) return;
  double next = 0.0;
  for (int x0 = last; x0 >= 0; x0 -= kChunk) {
    const int w = min(kChunk, nx - x0);
    if (x0 != last) {
      for (int r = 0; r < nr; ++r)
        if (lane < w) t[r][lane] = dst[(int64_t)r * nx + x0 + lane];
      __syncwarp();
    }
    if (mine) {
      int j = w - 1;
      if (x0 == last) {
        next = __dmul_rn(s.k, __dadd_rn(__dmul_rn(s.z, prev2), prev));
        t[lane][j--] = next;
      }
      for (; j >= 0; --j) {
        next = __dmul_rn(s.z, __dsub_rn(next, t[lane][j]));
        t[lane][j] = next;
      }
    }
    __syncwarp();
    for (int r = 0; r < nr; ++r)
      if (lane < w) dst[(int64_t)r * nx + x0 + lane] = t[r][lane];
    __syncwarp();
  }
}

// Along y (inner = nx) or z (inner = nx * ny), in place: thread = one line of n values `inner` apart; line l starts at
// (l / inner) * inner * n + l % inner, so adjacent threads take adjacent x.  Loads are issued kBatch at a time ahead
// of the recursion that consumes them.
constexpr int kBatch = 8;

__global__ void __launch_bounds__(128) bspline_line_kernel(double* __restrict__ coef, int64_t lines, int64_t inner,
                                                           int n) {
  pdl_wait();
  pdl_launch();
  const Spline s = spline_constants();
  const int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= lines || n == 1) return;
  double* p = coef + (l / inner) * inner * n + l % inner;
  double prev = causal_init(s, n, [&](int j) { return __dmul_rn(p[j * inner], s.gain); });
  double prev2 = 0.0;
  p[0] = prev;
  for (int j0 = 1; j0 < n; j0 += kBatch) {
    double v[kBatch];
#pragma unroll
    for (int b = 0; b < kBatch; ++b)
      if (j0 + b < n) v[b] = p[(j0 + b) * inner];
#pragma unroll
    for (int b = 0; b < kBatch; ++b)
      if (j0 + b < n) {
        const double c = __dadd_rn(__dmul_rn(v[b], s.gain), __dmul_rn(s.z, prev));
        p[(j0 + b) * inner] = c;
        prev2 = prev;
        prev = c;
      }
  }
  double next = __dmul_rn(s.k, __dadd_rn(__dmul_rn(s.z, prev2), prev));
  p[(int64_t)(n - 1) * inner] = next;
  for (int j0 = n - 2; j0 >= 0; j0 -= kBatch) {
    double v[kBatch];
#pragma unroll
    for (int b = 0; b < kBatch; ++b)
      if (j0 - b >= 0) v[b] = p[(j0 - b) * inner];
#pragma unroll
    for (int b = 0; b < kBatch; ++b)
      if (j0 - b >= 0) {
        next = __dmul_rn(s.z, __dsub_rn(next, v[b]));
        p[(j0 - b) * inner] = next;
      }
  }
}

// Taps f-1 .. f+2 of one axis, mirrored with period 2n - 2, and ITK's order-3 weights; an axis of extent 1 has one tap.
__device__ __forceinline__ void spline_axis(double c, int n, int tap[4], double wt[4]) {
  if (n == 1) {
    tap[0] = tap[1] = tap[2] = tap[3] = 0;
    wt[0] = 1.0, wt[1] = wt[2] = wt[3] = 0.0;
    return;
  }
  const double f = floor(c);
  const double w = __dsub_rn(c, f);
  const double sixth = 1.0 / 6.0;
  wt[3] = __dmul_rn(__dmul_rn(__dmul_rn(sixth, w), w), w);
  wt[0] = __dsub_rn(__dadd_rn(sixth, __dmul_rn(__dmul_rn(0.5, w), __dsub_rn(w, 1.0))), wt[3]);
  wt[2] = __dsub_rn(__dadd_rn(w, wt[0]), __dmul_rn(2.0, wt[3]));
  wt[1] = __dsub_rn(__dsub_rn(__dsub_rn(1.0, wt[0]), wt[2]), wt[3]);
  const int period = 2 * n - 2;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    int j = abs((int)f - 1 + t);
    if (j >= period) j -= period;
    if (j >= n) j = period - j;
    tap[t] = j;
  }
}

__device__ __forceinline__ double spline_sum(const double a[4], const double wt[4], bool single) {
  return single ? a[0]
                : __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(wt[0], a[0]), __dmul_rn(wt[1], a[1])),
                                      __dmul_rn(wt[2], a[2])),
                            __dmul_rn(wt[3], a[3]));
}

template <bool kVol>
__device__ __forceinline__ void bspline_voxel(const double* __restrict__ coef, const Map& m, const Ext& e, int row, int x,
                                              float dflt, float* __restrict__ out) {
  const int iy = row % e.out[1];
  const int rz = row / e.out[1];
  const int iz = kVol ? rz % e.out[2] : 0;
  const int64_t item = kVol ? rz / e.out[2] : rz;
  double c[3];
  const bool ok = cindex<kVol>(m, e, (double)x, (double)iy, (double)iz, c);
  float r = dflt;
  if (ok) {
    const int64_t plane = (int64_t)e.in[0] * e.in[1];
    const double* src = coef + item * plane * e.in[2];
    int tx[4], ty[4], tz[4];
    double wx[4], wy[4], wz[4];
    spline_axis(c[0], e.in[0], tx, wx);
    spline_axis(c[1], e.in[1], ty, wy);
    spline_axis(c[2], e.in[2], tz, wz);
    const bool sx = e.in[0] == 1, sy = e.in[1] == 1, sz = e.in[2] == 1;
    double az[4];
#pragma unroll
    for (int kz = 0; kz < (kVol ? 4 : 1); ++kz) {
      double ay[4];
#pragma unroll
      for (int ky = 0; ky < 4; ++ky) {
        const double* line = src + tz[kz] * plane + (int64_t)ty[ky] * e.in[0];
        double ax[4];
#pragma unroll
        for (int kx = 0; kx < 4; ++kx) ax[kx] = __ldg(line + tx[kx]);
        ay[ky] = spline_sum(ax, wx, sx);
      }
      az[kz] = spline_sum(ay, wy, sy);
    }
    r = __double2float_rn(kVol ? spline_sum(az, wz, sz) : az[0]);
  }
  out[(int64_t)row * e.out[0] + x] = r;
}

template <bool kVol>
__global__ void __launch_bounds__(128) resample_bspline_kernel(const double* __restrict__ coef, Map m, Ext e, int rows,
                                                               float dflt, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int row = blockIdx.x * kRows + threadIdx.y;
  const int x = blockIdx.y * 32 + threadIdx.x;
  if (row >= rows || x >= e.out[0]) return;
  bspline_voxel<kVol>(coef, m, e, row, x, dflt, out);
}

// The map is staged before the x test, so that every lane of the warp is present for it.
template <bool kVol>
__global__ void __launch_bounds__(128) resample_bspline_maps_kernel(const double* __restrict__ coef,
                                                                    const double* __restrict__ maps, Ext e, int rows,
                                                                    float dflt, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  __shared__ Map sm[kRows];
  const int row = blockIdx.x * kRows + threadIdx.y;
  const int x = blockIdx.y * 32 + threadIdx.x;
  if (row >= rows) return;
  const Map& m = stage_map(maps, e, row, &sm[threadIdx.y]);
  if (x >= e.out[0]) return;
  bspline_voxel<kVol>(coef, m, e, row, x, dflt, out);
}

// The linear entry point's validation, for the entry points that take a source and a target grid.
// With maps (device, items x 24) instead of map, the words are the caller's to keep finite: they are not read here.
static int check_grids(const char* what, const void* in, const void* out, int64_t items, int32_t rank,
                       const int32_t in_size[3], const int32_t out_size[3], const double map[24], Map& m, Ext& e,
                       int& rows, const double* maps = nullptr) {
  MPGAN_REQUIRE(in && out && in_size && out_size && (map || maps), MPGAN_ERR_SHAPE, "%s: null pointer", what);
  MPGAN_REQUIRE(items >= 1, MPGAN_ERR_SHAPE, "%s: items %lld (at least 1)", what, (long long)items);
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "%s: rank %d (2 or 3)", what, (int)rank);
  for (int k = 0; k < 3; ++k) {
    e.in[k] = in_size[k];
    e.out[k] = out_size[k];
    MPGAN_REQUIRE(e.in[k] >= 1 && e.in[k] <= kMaxExtent && e.out[k] >= 1 && e.out[k] <= kMaxExtent, MPGAN_ERR_SHAPE,
                  "%s: axis %c: input extent %d, output extent %d (each in [1, 2^22])", what, "xyz"[k], e.in[k],
                  e.out[k]);
  }
  if (maps) {
    MPGAN_REQUIRE(rank == 3 || (e.in[2] == 1 && e.out[2] == 1), MPGAN_ERR_SHAPE,
                  "%s: rank 2 with z extents %d, %d (must be 1)", what, e.in[2], e.out[2]);
  } else {
  for (int i = 0; i < 24; ++i)
    MPGAN_REQUIRE(isfinite(map[i]), MPGAN_ERR_SHAPE, "%s: map[%d] = %g is not finite", what, i, map[i]);
  for (int i = 0; i < 3; ++i) {
    m.oo[i] = map[i];
    m.oi[i] = map[12 + i];
  }
  for (int i = 0; i < 9; ++i) {
    m.m[i] = map[3 + i];
    m.n[i] = map[15 + i];
  }
  }
  if (rank == 2 && !maps) {
    MPGAN_REQUIRE(e.in[2] == 1 && e.out[2] == 1, MPGAN_ERR_SHAPE, "%s: rank 2 with z extents %d, %d (must be 1)", what,
                  e.in[2], e.out[2]);
    const double* mats[2] = {m.m, m.n};
    for (int t = 0; t < 2; ++t)
      MPGAN_REQUIRE(mats[t][2] == 0.0 && mats[t][5] == 0.0 && mats[t][6] == 0.0 && mats[t][7] == 0.0 && mats[t][8] == 1.0,
                    MPGAN_ERR_SHAPE, "%s: rank 2 needs the z row and column of %s to be the identity's", what,
                    t ? "N_in" : "M_out");
    MPGAN_REQUIRE(m.oo[2] == 0.0 && m.oi[2] == 0.0, MPGAN_ERR_SHAPE, "%s: rank 2 needs z origins 0, got %g and %g", what,
                  m.oo[2], m.oi[2]);
  }
  const int64_t row_len = (int64_t)e.out[1] * e.out[2];
  MPGAN_REQUIRE(items <= 0x7fffffffLL / row_len, MPGAN_ERR_SHAPE,
                "%s: %lld items of %lld output rows each exceed 2^31 - 1 rows", what, (long long)items,
                (long long)row_len);
  MPGAN_REQUIRE((double)items * e.in[0] * e.in[1] * e.in[2] < 0x1p62 && (double)items * e.out[0] * row_len < 0x1p62,
                MPGAN_ERR_SHAPE, "%s: tensor too large", what);
  rows = (int)(items * row_len);
  return 0;
}

}  // namespace resample
}  // namespace mpgan

extern "C" int mpgan_resample_nearest(const void* in, int32_t elem_bytes, int64_t items, int32_t rank,
                                      const int32_t in_size[3], const int32_t out_size[3], const double map[24],
                                      uint32_t default_bits, void* out, void* stream) {
  using namespace mpgan::resample;
  Map m;
  Ext e;
  int rows = 0;
  if (int rc = check_grids("resample_nearest", in, out, items, rank, in_size, out_size, map, m, e, rows)) return rc;
  MPGAN_REQUIRE(elem_bytes == 1 || elem_bytes == 4, MPGAN_ERR_SHAPE, "resample_nearest: elem_bytes %d (1 or 4)",
                (int)elem_bytes);
  const dim3 grid((unsigned)ceil_div(rows, kRows), (unsigned)ceil_div(e.out[0], 32 * kVox));
  const dim3 block(32, kRows);
  const cudaStream_t st = (cudaStream_t)stream;
  if (elem_bytes == 1) {
    const uint8_t d = (uint8_t)default_bits;
    if (rank == 3)
      launch_k(resample_nearest_kernel<uint8_t, true>, grid, block, 0, st, (const uint8_t*)in, m, e, rows, d,
               (uint8_t*)out);
    else
      launch_k(resample_nearest_kernel<uint8_t, false>, grid, block, 0, st, (const uint8_t*)in, m, e, rows, d,
               (uint8_t*)out);
  } else {
    if (rank == 3)
      launch_k(resample_nearest_kernel<uint32_t, true>, grid, block, 0, st, (const uint32_t*)in, m, e, rows,
               default_bits, (uint32_t*)out);
    else
      launch_k(resample_nearest_kernel<uint32_t, false>, grid, block, 0, st, (const uint32_t*)in, m, e, rows,
               default_bits, (uint32_t*)out);
  }
  MPGAN_CHECK_LAUNCH("resample_nearest_kernel");
  return 0;
}

extern "C" int mpgan_bspline_coefficients(const float* in, int64_t items, int32_t rank, const int32_t size[3],
                                          double* coef, void* stream) {
  using namespace mpgan::resample;
  MPGAN_REQUIRE(in && coef && size, MPGAN_ERR_SHAPE, "bspline_coefficients: null pointer");
  MPGAN_REQUIRE(items >= 1, MPGAN_ERR_SHAPE, "bspline_coefficients: items %lld (at least 1)", (long long)items);
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "bspline_coefficients: rank %d (2 or 3)", (int)rank);
  int n[3];
  for (int k = 0; k < 3; ++k) {
    n[k] = size[k];
    MPGAN_REQUIRE(n[k] >= 1 && n[k] <= kMaxExtent, MPGAN_ERR_SHAPE,
                  "bspline_coefficients: axis %c: extent %d (in [1, 2^22])", "xyz"[k], n[k]);
  }
  MPGAN_REQUIRE(rank == 3 || n[2] == 1, MPGAN_ERR_SHAPE, "bspline_coefficients: rank 2 with z extents %d (must be 1)",
                n[2]);
  int64_t lines = (int64_t)n[1] * n[2];   // the most lines of one item along any axis
  if ((int64_t)n[0] * n[2] > lines) lines = (int64_t)n[0] * n[2];
  if ((int64_t)n[0] * n[1] > lines) lines = (int64_t)n[0] * n[1];
  MPGAN_REQUIRE(items <= 0x7fffffffLL / lines, MPGAN_ERR_SHAPE,
                "bspline_coefficients: %lld items of up to %lld lines each exceed 2^31 - 1 rows", (long long)items,
                (long long)lines);
  MPGAN_REQUIRE((double)items * n[0] * n[1] * n[2] < 0x1p62, MPGAN_ERR_SHAPE, "bspline_coefficients: tensor too large");
  const uintptr_t voxels = (uintptr_t)items * n[0] * n[1] * n[2];
  const uintptr_t a = (uintptr_t)in, b = (uintptr_t)coef;
  MPGAN_REQUIRE(a + 4 * voxels <= b || b + 8 * voxels <= a, MPGAN_ERR_SHAPE, "bspline_coefficients: in and coef overlap");
  const cudaStream_t st = (cudaStream_t)stream;
  const int rows = (int)(items * n[1] * n[2]);
  launch_k(bspline_x_kernel, dim3((unsigned)ceil_div(rows, 128)), dim3(32, 4), 0, st, in, coef, n[0], rows);
  MPGAN_CHECK_LAUNCH("bspline_x_kernel");
  for (int axis = 1; axis < rank; ++axis) {
    const int64_t inner = axis == 1 ? (int64_t)n[0] : (int64_t)n[0] * n[1];
    const int64_t count = items * n[0] * n[1] * n[2] / n[axis];
    launch_k(bspline_line_kernel, dim3((unsigned)ceil_div(count, 128)), dim3(128), 0, st, coef, count, inner, n[axis]);
    MPGAN_CHECK_LAUNCH("bspline_line_kernel");
  }
  return 0;
}

extern "C" int mpgan_resample_bspline(const double* coef, int64_t items, int32_t rank, const int32_t in_size[3],
                                      const int32_t out_size[3], const double map[24], float default_value, float* out,
                                      void* stream) {
  using namespace mpgan::resample;
  Map m;
  Ext e;
  int rows = 0;
  if (int rc = check_grids("resample_bspline", coef, out, items, rank, in_size, out_size, map, m, e, rows)) return rc;
  const dim3 grid((unsigned)ceil_div(rows, kRows), (unsigned)ceil_div(e.out[0], 32));
  if (rank == 3)
    launch_k(resample_bspline_kernel<true>, grid, dim3(32, kRows), 0, (cudaStream_t)stream, coef, m, e, rows,
             default_value, out);
  else
    launch_k(resample_bspline_kernel<false>, grid, dim3(32, kRows), 0, (cudaStream_t)stream, coef, m, e, rows,
             default_value, out);
  MPGAN_CHECK_LAUNCH("resample_bspline_kernel");
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// The same three interpolations with one map per item read from device memory (a rigid transform composed with the
// target grid, mpgan_rigid_maps); the kernels above with the map staged in shared memory.
extern "C" int mpgan_resample_linear_maps(const float* in, int64_t items, int32_t rank, const int32_t in_size[3],
                                          const int32_t out_size[3], const double* maps, float default_value,
                                          float* out, void* stream) {
  using namespace mpgan::resample;
  Map m;
  Ext e;
  int rows = 0;
  if (int rc = check_grids("resample_linear_maps", in, out, items, rank, in_size, out_size, nullptr, m, e, rows, maps))
    return rc;
  const dim3 grid((unsigned)ceil_div(rows, kRows), (unsigned)ceil_div(e.out[0], 32 * kVox));
  const cudaStream_t st = (cudaStream_t)stream;
  if (rank == 3)
    launch_k(resample_linear_maps_kernel<true>, grid, dim3(32, kRows), 0, st, in, maps, e, rows, default_value, out);
  else
    launch_k(resample_linear_maps_kernel<false>, grid, dim3(32, kRows), 0, st, in, maps, e, rows, default_value, out);
  MPGAN_CHECK_LAUNCH("resample_linear_maps_kernel");
  return 0;
}

extern "C" int mpgan_resample_nearest_maps(const void* in, int32_t elem_bytes, int64_t items, int32_t rank,
                                           const int32_t in_size[3], const int32_t out_size[3], const double* maps,
                                           uint32_t default_bits, void* out, void* stream) {
  using namespace mpgan::resample;
  Map m;
  Ext e;
  int rows = 0;
  if (int rc = check_grids("resample_nearest_maps", in, out, items, rank, in_size, out_size, nullptr, m, e, rows, maps))
    return rc;
  MPGAN_REQUIRE(elem_bytes == 1 || elem_bytes == 4, MPGAN_ERR_SHAPE, "resample_nearest_maps: elem_bytes %d (1 or 4)",
                (int)elem_bytes);
  const dim3 grid((unsigned)ceil_div(rows, kRows), (unsigned)ceil_div(e.out[0], 32 * kVox));
  const dim3 block(32, kRows);
  const cudaStream_t st = (cudaStream_t)stream;
  if (elem_bytes == 1) {
    const uint8_t d = (uint8_t)default_bits;
    if (rank == 3)
      launch_k(resample_nearest_maps_kernel<uint8_t, true>, grid, block, 0, st, (const uint8_t*)in, maps, e, rows, d,
               (uint8_t*)out);
    else
      launch_k(resample_nearest_maps_kernel<uint8_t, false>, grid, block, 0, st, (const uint8_t*)in, maps, e, rows, d,
               (uint8_t*)out);
  } else {
    if (rank == 3)
      launch_k(resample_nearest_maps_kernel<uint32_t, true>, grid, block, 0, st, (const uint32_t*)in, maps, e, rows,
               default_bits, (uint32_t*)out);
    else
      launch_k(resample_nearest_maps_kernel<uint32_t, false>, grid, block, 0, st, (const uint32_t*)in, maps, e, rows,
               default_bits, (uint32_t*)out);
  }
  MPGAN_CHECK_LAUNCH("resample_nearest_maps_kernel");
  return 0;
}

extern "C" int mpgan_resample_bspline_maps(const double* coef, int64_t items, int32_t rank, const int32_t in_size[3],
                                           const int32_t out_size[3], const double* maps, float default_value,
                                           float* out, void* stream) {
  using namespace mpgan::resample;
  Map m;
  Ext e;
  int rows = 0;
  if (int rc = check_grids("resample_bspline_maps", coef, out, items, rank, in_size, out_size, nullptr, m, e, rows,
                           maps))
    return rc;
  const dim3 grid((unsigned)ceil_div(rows, kRows), (unsigned)ceil_div(e.out[0], 32));
  const cudaStream_t st = (cudaStream_t)stream;
  if (rank == 3)
    launch_k(resample_bspline_maps_kernel<true>, grid, dim3(32, kRows), 0, st, coef, maps, e, rows, default_value, out);
  else
    launch_k(resample_bspline_maps_kernel<false>, grid, dim3(32, kRows), 0, st, coef, maps, e, rows, default_value,
             out);
  MPGAN_CHECK_LAUNCH("resample_bspline_maps_kernel");
  return 0;
}
