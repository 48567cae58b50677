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

template <bool kVol>
__global__ void __launch_bounds__(128) resample_linear_kernel(const float* __restrict__ in, Map m, Ext e, int rows,
                                                              float dflt, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int row = blockIdx.x * kRows + threadIdx.y;   // (item * out_z + iz) * out_y + iy
  if (row >= rows) return;
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
