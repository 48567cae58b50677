// Rigid registration by Mattes mutual information (the semantics pinned in include/mpgan.h, restated in
// oracle/registration.py), and the separable Gaussian filter its pyramid smooths with.
//
// Gaussian: one launch per axis.  Along x a 128-thread block stages a 128-column chunk of one row plus its reflected
// halo in shared memory; along y and z one thread per output voxel, adjacent threads on adjacent x, so every load and
// store of a warp is coalesced.  Intermediates are fp64; the last pass rounds once to fp32.
//
// Metric: per item and per chunk of fixed-sample rows, in the warp-per-row layout of the resample kernels (a warp
// owns a row of samples, lanes take samples 32 apart).  Pass 1 accumulates the joint histogram as fixed-point int64
// (each Parzen weight rounded to a multiple of 2^-32) in shared memory and flushes it with integer atomics, so the
// histogram is exact and independent of order.  A one-CTA-per-item kernel turns it into -MI and the B x B table of
// log(p / p_m).  Pass 2 sums the P derivative terms per CTA in fp64 in a fixed order; a per-item kernel adds the CTA
// partials in chunk order.  Results are bit-identical run to run and do not depend on the rest of the batch: the
// chunking of an item depends on its shape only.
//
// State: kState fp64 words per item (layout below), updated in place by tiny per-item kernels (level start, optimiser
// step).  No call reads anything back to the host, and the launch count depends on the arguments only, so a whole
// registration can be captured in a CUDA graph; items that have stopped run the remaining iterations as no-ops.
#include <algorithm>

#include "common.cuh"

namespace mpgan {
namespace reg {

constexpr int kState = 96;
enum : int {
  kParam = 0,      // mu[6]
  kMap = 6,        // the 24-word map: o', M', o_moving, N_moving
  kDer = 30,       // 3 x (do[3], dM[9]): derivatives of o' and M' by each rotation angle
  kGrad = 66,      // gradient of -MI by mu[6]
  kPrev = 72,      // previous scaled gradient g_u[6]
  kStep = 78,      // step length lambda
  kRange = 80,     // fixed min, fixed max, moving min, moving max
  kCount = 84,     // the level's fixed samples
  kSum = 86,       // sum of the histogram (fixed point, as fp64)
  kScale = 88,     // scales of the rotation parameters for the level (physical shift of the samples)
};
enum : int { kRunning = -1, kConverged = 0, kIterations = 1, kOverlap = 2, kFlat = 3 };

constexpr int kMaxRadius = 64;
constexpr int kMaxBins = 128;
constexpr int kThreads = 256;          // metric passes: 8 warps
constexpr int kRowsPerCta = 32;        // sample rows per CTA (4 per warp) before the chunk count is capped
constexpr int kMaxChunks = 512;
constexpr int kMaxExtent = 1 << 22;

struct Taps {
  double w[2 * kMaxRadius + 1];
  int r;
};

struct Sizes {
  int f[3], m[3];   // fixed and moving extents, ITK order x, y, z
};

// ---- Gaussian filter ----------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect(int j, int n) {
  const int p = 2 * n;
  j %= p;
  if (j < 0) j += p;
  return j >= n ? p - 1 - j : j;
}

template <typename TIn>
__global__ void __launch_bounds__(128) gauss_x_kernel(const TIn* __restrict__ in, double* __restrict__ out, int nx,
                                                      int chunks, Taps t) {
  pdl_wait();
  pdl_launch();
  __shared__ double s[128 + 2 * kMaxRadius];
  const int64_t row = blockIdx.x / chunks;
  const int x0 = (int)(blockIdx.x % chunks) * 128;
  const TIn* src = in + row * nx;
  for (int i = threadIdx.x; i < 128 + 2 * t.r; i += 128) s[i] = (double)src[reflect(x0 - t.r + i, nx)];
  __syncthreads();
  const int x = x0 + threadIdx.x;
  if (x >= nx) return;
  double acc = __dmul_rn(t.w[0], s[threadIdx.x]);
  for (int k = 1; k <= 2 * t.r; ++k) acc = __dadd_rn(acc, __dmul_rn(t.w[k], s[threadIdx.x + k]));
  out[row * nx + x] = acc;
}

template <typename TOut>
__global__ void __launch_bounds__(128) gauss_line_kernel(const double* __restrict__ in, TOut* __restrict__ out,
                                                         int64_t total, int64_t inner, int n, Taps t) {
  pdl_wait();
  pdl_launch();
  const int64_t idx = (int64_t)blockIdx.x * 128 + threadIdx.x;
  if (idx >= total) return;
  const int64_t i = idx % inner, rest = idx / inner;
  const int j = (int)(rest % n);
  const double* base = in + (rest / n) * n * inner + i;
  double acc = __dmul_rn(t.w[0], base[(int64_t)reflect(j - t.r, n) * inner]);
  for (int k = 1; k <= 2 * t.r; ++k) acc = __dadd_rn(acc, __dmul_rn(t.w[k], base[(int64_t)reflect(j - t.r + k, n) * inner]));
  if constexpr (sizeof(TOut) == 4)
    out[idx] = __double2float_rn(acc);
  else
    out[idx] = acc;
}

// ---- transform ----------------------------------------------------------------------------------------------------
// sin and cos: 2 pi reduction in two parts, then Horner in r^2 with the Taylor coefficients (-1)^k / (2k+1)! and
// (-1)^k / (2k)!, each correctly rounded (the oracle's SIN_C / COS_C).
__constant__ double kSinC[14] = {0x1.0000000000000p+0,  -0x1.5555555555555p-3, 0x1.1111111111111p-7,
                                 -0x1.a01a01a01a01ap-13, 0x1.71de3a556c734p-19, -0x1.ae64567f544e4p-26,
                                 0x1.6124613a86d09p-33,  -0x1.ae7f3e733b81fp-41, 0x1.952c77030ad4ap-49,
                                 -0x1.2f49b46814157p-57, 0x1.71b8ef6dcf572p-66,  -0x1.761b41316381ap-75,
                                 0x1.3f3ccdd165fa9p-84,  -0x1.d1ab1c2dccea3p-94};
__constant__ double kCosC[15] = {0x1.0000000000000p+0,  -0x1.0000000000000p-1, 0x1.5555555555555p-5,
                                 -0x1.6c16c16c16c17p-10, 0x1.a01a01a01a01ap-16,  -0x1.27e4fb7789f5cp-22,
                                 0x1.1eed8eff8d898p-29,  -0x1.93974a8c07c9dp-37, 0x1.ae7f3e733b81fp-45,
                                 -0x1.6827863b97d97p-53, 0x1.e542ba4020225p-62,  -0x1.0ce396db7f853p-70,
                                 0x1.f2cf01972f578p-80,  -0x1.88e85fc6a4e5ap-89, 0x1.0a18a2635085dp-98};

__device__ void pinned_sincos(double t, double& s, double& c) {
  const double n = rint(__dmul_rn(t, 0x1.45f306dc9c883p-3));
  const double r = __dsub_rn(__dsub_rn(t, __dmul_rn(n, 0x1.921fb54442d18p+2)), __dmul_rn(n, 2.4492935982947064e-16));
  const double r2 = __dmul_rn(r, r);
  double a = kSinC[13];
  for (int k = 12; k >= 0; --k) a = __dadd_rn(kSinC[k], __dmul_rn(r2, a));
  double b = kCosC[14];
  for (int k = 13; k >= 0; --k) b = __dadd_rn(kCosC[k], __dmul_rn(r2, b));
  s = __dmul_rn(r, a);
  c = b;
}

struct M3 {
  double a[3][3];
};

__device__ M3 mul3(const M3& x, const M3& y) {
  M3 z;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j)
      z.a[i][j] = __dadd_rn(__dadd_rn(__dmul_rn(x.a[i][0], y.a[0][j]), __dmul_rn(x.a[i][1], y.a[1][j])),
                            __dmul_rn(x.a[i][2], y.a[2][j]));
  return z;
}

// The base map (o_fixed, M_fixed, o_moving, N_moving) and the fixed centre, passed by value.
struct Base {
  double map[24];
  double c[3];
};

// (o', M') of rm: M' = rm M_fixed, o' = (rm (o_fixed - c) + c) + t; with t == nullptr, o' = rm (o_fixed - c).
__device__ void affine(const M3& rm, const Base& b, const double* t, double* o_out, double* m_out) {
  M3 mf;
  double d[3];
  for (int k = 0; k < 3; ++k) {
    d[k] = __dsub_rn(b.map[k], b.c[k]);
    for (int j = 0; j < 3; ++j) mf.a[k][j] = b.map[3 + 3 * k + j];
  }
  const M3 mm = mul3(rm, mf);
  for (int k = 0; k < 3; ++k) {
    const double e = __dadd_rn(__dadd_rn(__dmul_rn(rm.a[k][0], d[0]), __dmul_rn(rm.a[k][1], d[1])),
                               __dmul_rn(rm.a[k][2], d[2]));
    o_out[k] = t ? __dadd_rn(__dadd_rn(e, b.c[k]), t[k]) : e;
    for (int j = 0; j < 3; ++j) m_out[3 * k + j] = mm.a[k][j];
  }
}

// The map of parameters mu into map[24] and, when der != nullptr, the rotation-derivative maps into der[36].
__device__ void compose(const double* mu, int rank, const Base& b, double* map, double* der) {
  M3 r, dr[3];
  int nrot;
  double t[3];
  if (rank == 2) {
    double s, c;
    pinned_sincos(mu[0], s, c);
    r = M3{{{c, -s, 0.0}, {s, c, 0.0}, {0.0, 0.0, 1.0}}};
    dr[0] = M3{{{-s, -c, 0.0}, {c, -s, 0.0}, {0.0, 0.0, 0.0}}};
    nrot = 1;
    t[0] = mu[1], t[1] = mu[2], t[2] = 0.0;
  } else {
    double sx, cx, sy, cy, sz, cz;
    pinned_sincos(mu[0], sx, cx);
    pinned_sincos(mu[1], sy, cy);
    pinned_sincos(mu[2], sz, cz);
    const M3 rx{{{1.0, 0.0, 0.0}, {0.0, cx, -sx}, {0.0, sx, cx}}};
    const M3 ry{{{cy, 0.0, sy}, {0.0, 1.0, 0.0}, {-sy, 0.0, cy}}};
    const M3 rz{{{cz, -sz, 0.0}, {sz, cz, 0.0}, {0.0, 0.0, 1.0}}};
    const M3 drx{{{0.0, 0.0, 0.0}, {0.0, -sx, -cx}, {0.0, cx, -sx}}};
    const M3 dry{{{-sy, 0.0, cy}, {0.0, 0.0, 0.0}, {-cy, 0.0, -sy}}};
    const M3 drz{{{-sz, -cz, 0.0}, {cz, -sz, 0.0}, {0.0, 0.0, 0.0}}};
    const M3 zx = mul3(rz, rx);
    r = mul3(zx, ry);
    dr[0] = mul3(mul3(rz, drx), ry);
    dr[1] = mul3(zx, dry);
    dr[2] = mul3(mul3(drz, rx), ry);
    nrot = 3;
    t[0] = mu[3], t[1] = mu[4], t[2] = mu[5];
  }
  affine(r, b, t, map, map + 3);
  for (int i = 12; i < 24; ++i) map[i] = b.map[i];
  if (der)
    for (int j = 0; j < nrot; ++j) affine(dr[j], b, nullptr, der + 12 * j, der + 12 * j + 3);
}

__global__ void rigid_maps_kernel(const double* __restrict__ params, int items, int rank, Base b,
                                  double* __restrict__ maps) {
  pdl_wait();
  pdl_launch();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= items) return;
  const int P = rank == 3 ? 6 : 3;
  double mu[6];
  for (int j = 0; j < P; ++j) mu[j] = params[(int64_t)i * P + j];
  compose(mu, rank, b, maps + (int64_t)i * 24, nullptr);
}

// Level start.  first: mu = initial (device, items x P) or t0 in the translations; every item runs.  Later levels:
// items that failed (overlap, flat) stay as they are, the others run again.  Step, previous gradient and map reset.
__global__ void rigid_level_kernel(double* __restrict__ state, int* __restrict__ status, int items, int rank, Base b,
                                   const double* __restrict__ initial, double t0x, double t0y, double t0z, int first,
                                   double step) {
  pdl_wait();
  pdl_launch();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= items) return;
  const int P = rank == 3 ? 6 : 3;
  double* s = state + (int64_t)i * kState;
  if (first) {
    for (int j = 0; j < 6; ++j) s[kParam + j] = 0.0;
    if (initial) {
      for (int j = 0; j < P; ++j) s[kParam + j] = initial[(int64_t)i * P + j];
    } else {
      s[kParam + P - rank] = t0x;
      s[kParam + P - rank + 1] = t0y;
      if (rank == 3) s[kParam + 5] = t0z;
    }
    status[i] = kRunning;
  } else if (status[i] < kOverlap) {
    status[i] = kRunning;
  }
  s[kStep] = step;
  for (int j = 0; j < 6; ++j) s[kPrev + j] = 0.0;
  compose(s + kParam, rank, b, s + kMap, s + kDer);
}

// One regular-step gradient-descent step in scaled parameters u = scale * mu (include/mpgan.h).
__global__ void rigid_step_kernel(double* __restrict__ state, int* __restrict__ status, int items, int rank, Base b,
                                  double min_step, int last) {
  pdl_wait();
  pdl_launch();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= items || status[i] != kRunning) return;
  const int P = rank == 3 ? 6 : 3, nrot = rank == 3 ? 3 : 1;
  double* s = state + (int64_t)i * kState;
  double sc[6], gu[6], dot = 0.0, n2 = 0.0;
  for (int j = 0; j < P; ++j) sc[j] = j < nrot ? s[kScale + j] : 1.0;
  for (int j = 0; j < P; ++j) {
    gu[j] = __ddiv_rn(s[kGrad + j], sc[j]);
    dot = __dadd_rn(dot, __dmul_rn(gu[j], s[kPrev + j]));
  }
  double step = s[kStep];
  if (dot < 0.0) step = __dmul_rn(step, 0.5);
  s[kStep] = step;
  if (step < min_step) {
    status[i] = kConverged;
    return;
  }
  for (int j = 0; j < P; ++j) n2 = __dadd_rn(n2, __dmul_rn(gu[j], gu[j]));
  const double nrm = __dsqrt_rn(n2);
  if (!(nrm > 0.0)) {
    status[i] = kConverged;
    return;
  }
  for (int j = 0; j < P; ++j) {
    s[kParam + j] = __dsub_rn(s[kParam + j], __ddiv_rn(__ddiv_rn(__dmul_rn(step, gu[j]), nrm), sc[j]));
    s[kPrev + j] = gu[j];
  }
  compose(s + kParam, rank, b, s + kMap, s + kDer);
  if (last) status[i] = kIterations;
}

// ---- metric -------------------------------------------------------------------------------------------------------
struct Map {
  double oo[3], m[9], oi[3], n[9];
};

// Moving-image sample at fixed index (fx, fy, fz): the resample kernels' continuous index, inside test and linear
// corners; value in fp64 (not rounded).  b: base corner, s: neighbour steps (0 at weight 0), d: weights.
struct Corner {
  int64_t off, sy, sz;
  int sx;
  double d[3];
};

template <bool kVol>
__device__ __forceinline__ bool locate(const Map& m, const int* n, double fx, double fy, double fz, Corner& k) {
  double p[3], q[3], c[3];
#pragma unroll
  for (int a = 0; a < (kVol ? 3 : 2); ++a) {
    p[a] = __dadd_rn(__dadd_rn(m.oo[a], __dmul_rn(m.m[3 * a], fx)), __dmul_rn(m.m[3 * a + 1], fy));
    if (kVol) p[a] = __dadd_rn(p[a], __dmul_rn(m.m[3 * a + 2], fz));
    q[a] = __dsub_rn(p[a], m.oi[a]);
  }
#pragma unroll
  for (int a = 0; a < (kVol ? 3 : 2); ++a) {
    c[a] = __dadd_rn(__dmul_rn(m.n[3 * a], q[0]), __dmul_rn(m.n[3 * a + 1], q[1]));
    if (kVol) c[a] = __dadd_rn(c[a], __dmul_rn(m.n[3 * a + 2], q[2]));
  }
  if (!kVol) c[2] = 0.0;
  bool ok = true;
  int b[3], s[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    ok = ok && c[a] >= -0.5 && c[a] < (double)n[a] - 0.5;
    const double f = ok ? fmax(floor(c[a]), 0.0) : 0.0;
    const double dd = ok ? __dsub_rn(c[a], f) : 0.0;
    b[a] = (int)f;
    k.d[a] = dd > 0.0 ? dd : 0.0;
    s[a] = k.d[a] > 0.0 && b[a] + 1 < n[a] ? 1 : 0;
  }
  const int64_t plane = (int64_t)n[0] * n[1];
  k.off = ok ? ((int64_t)b[2] * n[1] + b[1]) * n[0] + b[0] : 0;
  k.sx = s[0];
  k.sy = (int64_t)s[1] * n[0];
  k.sz = s[2] * plane;
  return ok;
}

__device__ __forceinline__ double lerp(double a, double b, double d) {
  return __dadd_rn(a, __dmul_rn(__dsub_rn(b, a), d));
}

template <bool kVol>
__device__ __forceinline__ double interp(const float* __restrict__ src, const Corner& k) {
  const float* p0 = src + k.off;
  const double a0 = __ldg(p0), a1 = __ldg(p0 + k.sx), a2 = __ldg(p0 + k.sy), a3 = __ldg(p0 + k.sy + k.sx);
  const bool ux = k.d[0] > 0.0, uy = k.d[1] > 0.0;
  const double v00 = ux ? lerp(a0, a1, k.d[0]) : a0;
  const double v01 = ux ? lerp(a2, a3, k.d[0]) : a2;
  double r = uy ? lerp(v00, v01, k.d[1]) : v00;
  if (kVol && k.d[2] > 0.0) {
    const float* p1 = p0 + k.sz;
    const double a4 = __ldg(p1), a5 = __ldg(p1 + k.sx), a6 = __ldg(p1 + k.sy), a7 = __ldg(p1 + k.sy + k.sx);
    const double v10 = ux ? lerp(a4, a5, k.d[0]) : a4;
    const double v11 = ux ? lerp(a6, a7, k.d[0]) : a6;
    r = lerp(r, uy ? lerp(v10, v11, k.d[1]) : v10, k.d[2]);
  }
  return r;
}

__device__ __forceinline__ double bspline3(double u) {
  const double a = fabs(u);
  if (a < 1.0) {
    const double a2 = __dmul_rn(a, a);
    return __dadd_rn(__dsub_rn(2.0 / 3.0, a2), __dmul_rn(0.5, __dmul_rn(a2, a)));
  }
  if (a < 2.0) {
    const double b = __dsub_rn(2.0, a);
    return __ddiv_rn(__dmul_rn(__dmul_rn(b, b), b), 6.0);
  }
  return 0.0;
}

__device__ __forceinline__ double bspline3_deriv(double u) {
  const double a = fabs(u);
  if (a < 1.0) return __dmul_rn(u, __dsub_rn(__dmul_rn(1.5, a), 2.0));
  if (a < 2.0) {
    const double b = __dsub_rn(2.0, a);
    return copysign(__dmul_rn(0.5, __dmul_rn(b, b)), -u);
  }
  return 0.0;
}

__device__ __forceinline__ int bin_of(double xi, int bins) {
  return (int)fmin(fmax(floor(xi), 2.0), (double)(bins - 3));
}

__device__ __forceinline__ bool skip(int st, int only_running) {
  return only_running ? st != kRunning : st >= kOverlap;
}

struct Level {
  int shrink, bins, sx, rows;   // sample stride, bins, samples per row, sample rows per item
};

__device__ __forceinline__ void sample_row(const Level& L, const Sizes& z, int r, int& iy, int& iz) {
  const int sy = (z.f[1] + L.shrink - 1) / L.shrink;
  iy = (r % sy) * L.shrink;
  iz = (r / sy) * L.shrink;
}

// Per item (blockIdx.y) and chunk: fixed min / max over the level's samples, the sample count, and the moving image's
// min / max.  Extremes are reduced as order-preserving keys (key_of) with integer atomics: exact and order-free.
// keys: items x {max fixed, ~min fixed, max moving, ~min moving}; counts: items.
__global__ void __launch_bounds__(kThreads) mattes_range_kernel(const float* __restrict__ fixed,
                                                                const float* __restrict__ moving,
                                                                const uint8_t* __restrict__ mask, Sizes z, Level L,
                                                                unsigned* __restrict__ keys,
                                                                unsigned long long* __restrict__ counts,
                                                                unsigned long long* __restrict__ moments) {
  pdl_wait();
  pdl_launch();
  const int64_t item = blockIdx.y;
  const int64_t nf = (int64_t)z.f[0] * z.f[1] * z.f[2], nm = (int64_t)z.m[0] * z.m[1] * z.m[2];
  unsigned hi = 0, nlo = 0, cnt = 0;
  long long mo[6] = {0, 0, 0, 0, 0, 0};   // xx, yy, zz, xy, xz, yz of (2 i - (n - 1)), exact
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  if (blockIdx.z == 0) {
    const int64_t total = (int64_t)L.rows * L.sx;
    const float* f = fixed + item * nf;
    const uint8_t* mk = mask ? mask + item * nf : nullptr;
    for (int64_t s = (int64_t)blockIdx.x * kThreads + threadIdx.x; s < total; s += stride) {
      int iy, iz;
      sample_row(L, z, (int)(s / L.sx), iy, iz);
      const int ix = (int)(s % L.sx) * L.shrink;
      const int64_t v = ((int64_t)iz * z.f[1] + iy) * z.f[0] + ix;
      if (mk && !mk[v]) continue;
      const unsigned k = key_of(f[v]);
      hi = max(hi, k);
      nlo = max(nlo, ~k);
      ++cnt;
      const long long a = 2LL * ix - (z.f[0] - 1), b = 2LL * iy - (z.f[1] - 1), c = 2LL * iz - (z.f[2] - 1);
      mo[0] += a * a, mo[1] += b * b, mo[2] += c * c, mo[3] += a * b, mo[4] += a * c, mo[5] += b * c;
    }
  } else {
    const float* m = moving + item * nm;
    for (int64_t v = (int64_t)blockIdx.x * kThreads + threadIdx.x; v < nm; v += stride) {
      const unsigned k = key_of(m[v]);
      hi = max(hi, k);
      nlo = max(nlo, ~k);
    }
  }
  hi = __reduce_max_sync(0xffffffffu, hi);
  nlo = __reduce_max_sync(0xffffffffu, nlo);
  cnt = __reduce_add_sync(0xffffffffu, cnt);
#pragma unroll
  for (int j = 0; j < 6; ++j)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mo[j] += __shfl_xor_sync(0xffffffffu, mo[j], o);
  if ((threadIdx.x & 31) == 0) {
    unsigned* k = keys + item * 4 + 2 * blockIdx.z;
    if (hi) atomicMax(k, hi);
    if (nlo) atomicMax(k + 1, nlo);
    if (cnt) atomicAdd(counts + item, (unsigned long long)cnt);
    for (int j = 0; j < 6; ++j)   // two's complement: the unsigned sum of the signed terms is exact
      if (mo[j]) atomicAdd(moments + item * 6 + j, (unsigned long long)mo[j]);
  }
}

// Per item: the ranges into the state; flat (or NaN / inf) ranges set status flat, no samples sets overlap.
// The rotation scales: with S the exact index moments and M = M_fixed, C = (M S) M^T; v_k = C_kk / (4 n) is the mean
// squared physical offset of the samples from the grid centre along axis k, and the scale of the rotation about axis
// a is sqrt of the sum of the other two v (rank 2: the rotation about z, sqrt(v_x + v_y)), at least min_scale.
struct M9 {
  double a[9];
};

__global__ void mattes_range_finalize_kernel(const unsigned* __restrict__ keys,
                                             const unsigned long long* __restrict__ counts,
                                             const unsigned long long* __restrict__ moments, int items, int rank,
                                             M9 mf, double min_scale, double* __restrict__ state,
                                             int* __restrict__ status) {
  pdl_wait();
  pdl_launch();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= items) return;
  double* s = state + (int64_t)i * kState;
  const unsigned* k = keys + (int64_t)i * 4;
  const unsigned long long n = counts[i];
  const double fmin = n ? (double)value_of(~k[1]) : __longlong_as_double(0x7ff8000000000000LL);
  const double fmax = n ? (double)value_of(k[0]) : fmin;
  const double mmin = (double)value_of(~k[3]), mmax = (double)value_of(k[2]);
  s[kRange + 0] = fmin, s[kRange + 1] = fmax, s[kRange + 2] = mmin, s[kRange + 3] = mmax;
  s[kCount] = (double)n;
  const long long* mo = reinterpret_cast<const long long*>(moments) + (int64_t)i * 6;
  double S[9];
  S[0] = __ll2double_rn(mo[0]), S[4] = __ll2double_rn(mo[1]), S[8] = __ll2double_rn(mo[2]);
  S[1] = S[3] = __ll2double_rn(mo[3]), S[2] = S[6] = __ll2double_rn(mo[4]), S[5] = S[7] = __ll2double_rn(mo[5]);
  double v[3];
  for (int k = 0; k < 3; ++k) {   // row k of M S, then its product with row k of M
    double t[3];
    for (int j = 0; j < 3; ++j)
      t[j] = __dadd_rn(__dadd_rn(__dmul_rn(mf.a[3 * k], S[j]), __dmul_rn(mf.a[3 * k + 1], S[3 + j])),
                       __dmul_rn(mf.a[3 * k + 2], S[6 + j]));
    const double c = __dadd_rn(__dadd_rn(__dmul_rn(t[0], mf.a[3 * k]), __dmul_rn(t[1], mf.a[3 * k + 1])),
                               __dmul_rn(t[2], mf.a[3 * k + 2]));
    v[k] = n ? __ddiv_rn(c, __dmul_rn(4.0, (double)n)) : 0.0;
  }
  const int nrot = rank == 3 ? 3 : 1;
  for (int a = 0; a < nrot; ++a) {
    const int ax = rank == 3 ? a : 2;
    const double sum = ax == 0 ? __dadd_rn(v[1], v[2]) : ax == 1 ? __dadd_rn(v[0], v[2]) : __dadd_rn(v[0], v[1]);
    s[kScale + a] = ::fmax(__dsqrt_rn(sum), min_scale);   // the local fmax above shadows the function
  }
  if (status[i] >= kOverlap) return;
  const bool ok = fmax > fmin && mmax > mmin && isfinite(fmin) && isfinite(fmax) && isfinite(mmin) && isfinite(mmax);
  if (!ok) status[i] = n ? kFlat : kOverlap;
}

// Central differences of the moving image along x, y, z (one-sided at the borders, 0 along an extent of 1), fp32,
// planar: grad[item][axis][voxel].
__global__ void __launch_bounds__(128) moving_gradient_kernel(const float* __restrict__ m, Sizes z, int64_t total,
                                                              float* __restrict__ grad) {
  pdl_wait();
  pdl_launch();
  const int64_t idx = (int64_t)blockIdx.x * 128 + threadIdx.x;
  if (idx >= total) return;
  const int64_t nm = (int64_t)z.m[0] * z.m[1] * z.m[2];
  const int64_t item = idx / nm, v = idx % nm;
  int c[3] = {(int)(v % z.m[0]), (int)((v / z.m[0]) % z.m[1]), (int)(v / ((int64_t)z.m[0] * z.m[1]))};
  const int64_t step[3] = {1, z.m[0], (int64_t)z.m[0] * z.m[1]};
  for (int a = 0; a < 3; ++a) {
    const int n = z.m[a];
    float g = 0.0f;
    if (n > 1) {
      const float* p = m + idx;
      if (c[a] == 0)
        g = __fsub_rn(p[step[a]], p[0]);
      else if (c[a] == n - 1)
        g = __fsub_rn(p[0], p[-step[a]]);
      else
        g = __fmul_rn(__fsub_rn(p[step[a]], p[-step[a]]), 0.5f);
    }
    grad[(item * 3 + a) * nm + v] = g;
  }
}

__device__ __forceinline__ void load_map(const double* __restrict__ s, Map* sm) {
  if (threadIdx.x < 24) reinterpret_cast<double*>(sm)[threadIdx.x] = s[kMap + threadIdx.x];
}

// Pass 1: the fixed-point joint histogram of the item's samples in this chunk.  hist: items x B x B (zeroed by the
// caller), inside: items.  A warp whose 32 samples all fall into one (fixed bin, moving base bin) adds their weights
// with one shared atomic per bin (background piles into one bin); otherwise every sample adds its own four.
template <bool kVol>
__global__ void __launch_bounds__(kThreads) mattes_hist_kernel(const float* __restrict__ fixed,
                                                               const float* __restrict__ moving,
                                                               const uint8_t* __restrict__ mask, Sizes z, Level L,
                                                               const double* __restrict__ state,
                                                               const int* __restrict__ status, int only_running,
                                                               unsigned long long* __restrict__ hist,
                                                               unsigned long long* __restrict__ inside) {
  pdl_wait();
  pdl_launch();
  extern __shared__ unsigned long long sh[];
  __shared__ Map sm;
  const int64_t item = blockIdx.y;
  if (skip(status[item], only_running)) return;
  const int B = L.bins, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < B * B; i += kThreads) sh[i] = 0;
  const double* st = state + item * kState;
  load_map(st, &sm);
  __syncthreads();
  const double fmin = st[kRange], mmin = st[kRange + 2];
  const double df = __ddiv_rn(__dsub_rn(st[kRange + 1], fmin), (double)(B - 4));
  const double dm = __ddiv_rn(__dsub_rn(st[kRange + 3], mmin), (double)(B - 4));
  const int64_t nf = (int64_t)z.f[0] * z.f[1] * z.f[2];
  const float* f = fixed + item * nf;
  const uint8_t* mk = mask ? mask + item * nf : nullptr;
  const float* mv = moving + item * ((int64_t)z.m[0] * z.m[1] * z.m[2]);
  unsigned cnt = 0;
  for (int r = blockIdx.x * (kThreads / 32) + warp; r < L.rows; r += gridDim.x * (kThreads / 32)) {
    int iy, iz;
    sample_row(L, z, r, iy, iz);
    const int64_t row = ((int64_t)iz * z.f[1] + iy) * z.f[0];
    for (int x0 = 0; x0 < L.sx; x0 += 32) {
      const int ix = (x0 + lane) * L.shrink;
      bool ok = x0 + lane < L.sx && (!mk || mk[row + ix]);
      Corner k;
      ok = ok && locate<kVol>(sm, z.m, (double)ix, (double)iy, (double)iz, k);
      int key = -1 - lane;   // unique per lane when invalid
      unsigned long long q[4] = {0, 0, 0, 0};
      int fb = 0, mb = 0;
      if (ok) {
        const double v = interp<kVol>(mv, k);
        fb = bin_of(__dadd_rn(__ddiv_rn(__dsub_rn((double)f[row + ix], fmin), df), 2.0), B);
        const double xm = __dadd_rn(__ddiv_rn(__dsub_rn(v, mmin), dm), 2.0);
        mb = bin_of(xm, B);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          q[j] = (unsigned long long)__double2ll_rn(__dmul_rn(bspline3(__dsub_rn((double)(mb - 1 + j), xm)), 0x1p32));
        key = fb * B + mb;
        ++cnt;
      }
      int same = 0;
      __match_all_sync(0xffffffffu, key, &same);
      if (same) {   // every lane valid and in one bin pair: weights < 2^32, summed as 16-bit halves
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(q[j] & 0xffffu));
          const unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)(q[j] >> 16));
          if (lane == 0) atomicAdd(&sh[fb * B + mb - 1 + j], ((unsigned long long)hi << 16) + lo);
        }
      } else if (ok) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (q[j]) atomicAdd(&sh[fb * B + mb - 1 + j], q[j]);
      }
    }
  }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if (lane == 0 && cnt) atomicAdd(inside + item, (unsigned long long)cnt);
  __syncthreads();
  unsigned long long* g = hist + item * B * B;
  for (int i = threadIdx.x; i < B * B; i += kThreads)
    if (sh[i]) atomicAdd(g + i, sh[i]);
}

// One CTA (128 threads) per item: -MI into metric, log(H / H_m) into lt (items x B x B), the histogram sum into the
// state.  Too few samples inside (4 inside < fixed samples, or none) sets status overlap and metric NaN.
__global__ void __launch_bounds__(128) mattes_finalize_kernel(const unsigned long long* __restrict__ hist,
                                                              const unsigned long long* __restrict__ inside, int bins,
                                                              double* __restrict__ state, int* __restrict__ status,
                                                              int only_running, double* __restrict__ metric,
                                                              double* __restrict__ lt) {
  pdl_wait();
  pdl_launch();
  __shared__ long long hm[kMaxBins], hf[kMaxBins];
  __shared__ double rows[kMaxBins];
  const int64_t item = blockIdx.x;
  if (skip(status[item], only_running)) return;
  double* s = state + item * kState;
  const unsigned long long n = inside[item];
  if (n == 0 || 4.0 * (double)n < s[kCount]) {
    __syncthreads();
    if (threadIdx.x == 0) {
      status[item] = kOverlap;
      metric[item] = __longlong_as_double(0x7ff8000000000000LL);
    }
    return;
  }
  const int B = bins;
  const long long* h = reinterpret_cast<const long long*>(hist) + item * B * B;
  for (int i = threadIdx.x; i < B; i += 128) {
    long long a = 0, b = 0;
    for (int j = 0; j < B; ++j) a += h[i * B + j], b += h[j * B + i];
    hf[i] = a, hm[i] = b;
  }
  __syncthreads();
  long long tot = 0;
  for (int i = 0; i < B; ++i) tot += hf[i];
  const double S = __ll2double_rn(tot);
  double* L = lt + item * B * B;
  for (int i = threadIdx.x; i < B; i += 128) {
    const double pf = __ddiv_rn(__ll2double_rn(hf[i]), S);
    double acc = 0.0;
    for (int j = 0; j < B; ++j) {
      const long long v = h[i * B + j];
      double l = 0.0;
      if (v > 0) {
        const double p = __ddiv_rn(__ll2double_rn(v), S), pm = __ddiv_rn(__ll2double_rn(hm[j]), S);
        acc = __dadd_rn(acc, __dmul_rn(p, log(__ddiv_rn(p, __dmul_rn(pf, pm)))));
        l = log(__ddiv_rn(__ll2double_rn(v), __ll2double_rn(hm[j])));
      }
      L[i * B + j] = l;
    }
    rows[i] = acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double mi = 0.0;
    for (int i = 0; i < B; ++i) mi = __dadd_rn(mi, rows[i]);
    metric[item] = -mi;
    s[kSum] = S;
  }
}

// Pass 2: per CTA, the P sums  sum_samples a * (grad M . dq/dmu_j)  with a = sum_k beta3'(k - xi_m) L[f][k], in fp64,
// reduced across the CTA in a fixed order into partial[item][chunk][6].
template <bool kVol>
__global__ void __launch_bounds__(kThreads) mattes_grad_kernel(const float* __restrict__ fixed,
                                                               const float* __restrict__ moving,
                                                               const float* __restrict__ grad,
                                                               const uint8_t* __restrict__ mask, Sizes z, Level L,
                                                               const double* __restrict__ state,
                                                               const int* __restrict__ status,
                                                               const double* __restrict__ lt,
                                                               double* __restrict__ partial) {
  pdl_wait();
  pdl_launch();
  extern __shared__ double tab[];
  __shared__ Map sm;
  __shared__ double der[36];
  __shared__ double red[kThreads / 32][6];
  const int64_t item = blockIdx.y;
  if (status[item] != kRunning) return;
  const int B = L.bins, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double* st = state + item * kState;
  for (int i = threadIdx.x; i < B * B; i += kThreads) tab[i] = lt[item * B * B + i];
  load_map(st, &sm);
  if (threadIdx.x < 36) der[threadIdx.x] = st[kDer + threadIdx.x];
  __syncthreads();
  const double fmin = st[kRange], mmin = st[kRange + 2];
  const double df = __ddiv_rn(__dsub_rn(st[kRange + 1], fmin), (double)(B - 4));
  const double dm = __ddiv_rn(__dsub_rn(st[kRange + 3], mmin), (double)(B - 4));
  const int64_t nf = (int64_t)z.f[0] * z.f[1] * z.f[2], nm = (int64_t)z.m[0] * z.m[1] * z.m[2];
  const float* f = fixed + item * nf;
  const uint8_t* mk = mask ? mask + item * nf : nullptr;
  const float* mv = moving + item * nm;
  const float* gx = grad + item * 3 * nm;
  const int nrot = kVol ? 3 : 1;
  double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  for (int r = blockIdx.x * (kThreads / 32) + warp; r < L.rows; r += gridDim.x * (kThreads / 32)) {
    int iy, iz;
    sample_row(L, z, r, iy, iz);
    const int64_t row = ((int64_t)iz * z.f[1] + iy) * z.f[0];
    for (int x0 = 0; x0 < L.sx; x0 += 32) {
      const int ix = (x0 + lane) * L.shrink;
      if (x0 + lane >= L.sx || (mk && !mk[row + ix])) continue;
      Corner k;
      if (!locate<kVol>(sm, z.m, (double)ix, (double)iy, (double)iz, k)) continue;
      const double v = interp<kVol>(mv, k);
      const int fb = bin_of(__dadd_rn(__ddiv_rn(__dsub_rn((double)f[row + ix], fmin), df), 2.0), B);
      const double xm = __dadd_rn(__ddiv_rn(__dsub_rn(v, mmin), dm), 2.0);
      const int mb = bin_of(xm, B);
      double a = 0.0;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        a = __dadd_rn(a, __dmul_rn(bspline3_deriv(__dsub_rn((double)(mb - 1 + j), xm)), tab[fb * B + mb - 1 + j]));
      if (a == 0.0) continue;
      double gi[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) gi[c] = (kVol || c < 2) ? interp<kVol>(gx + c * nm, k) : 0.0;
      double gp[3];
#pragma unroll
      for (int c = 0; c < 3; ++c)
        gp[c] = __dadd_rn(__dadd_rn(__dmul_rn(sm.n[c], gi[0]), __dmul_rn(sm.n[3 + c], gi[1])), __dmul_rn(sm.n[6 + c], gi[2]));
      const double fx = (double)ix, fy = (double)iy, fz = (double)iz;
      for (int j = 0; j < nrot; ++j) {
        const double* d = der + 12 * j;
        double col = 0.0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const double jc = __dadd_rn(__dadd_rn(__dadd_rn(d[c], __dmul_rn(d[3 + 3 * c], fx)), __dmul_rn(d[4 + 3 * c], fy)),
                                      __dmul_rn(d[5 + 3 * c], fz));
          col = __dadd_rn(col, __dmul_rn(gp[c], jc));
        }
        acc[j] = __dadd_rn(acc[j], __dmul_rn(a, col));
      }
#pragma unroll
      for (int c = 0; c < (kVol ? 3 : 2); ++c) acc[nrot + c] = __dadd_rn(acc[nrot + c], __dmul_rn(a, gp[c]));
    }
  }
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double v = acc[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = __dadd_rn(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (lane == 0) red[warp][j] = v;
  }
  __syncthreads();
  if (threadIdx.x < 6) {
    double v = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) v = __dadd_rn(v, red[w][threadIdx.x]);
    partial[(item * gridDim.x + blockIdx.x) * 6 + threadIdx.x] = v;
  }
}

// Per item: the CTA partials in chunk order, scaled by 2^32 / (sum H * delta_m), into the state's gradient.
__global__ void mattes_grad_reduce_kernel(const double* __restrict__ partial, int chunks, int items,
                                          double* __restrict__ state, const int* __restrict__ status, int bins) {
  pdl_wait();
  pdl_launch();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= items || status[i] != kRunning) return;
  double* s = state + (int64_t)i * kState;
  const double dm = __ddiv_rn(__dsub_rn(s[kRange + 3], s[kRange + 2]), (double)(bins - 4));
  const double scale = __ddiv_rn(0x1p32, __dmul_rn(s[kSum], dm));
  for (int j = 0; j < 6; ++j) {
    double v = 0.0;
    for (int c = 0; c < chunks; ++c) v = __dadd_rn(v, partial[((int64_t)i * chunks + c) * 6 + j]);
    s[kGrad + j] = __dmul_rn(v, scale);
  }
}

// ---- host helpers -------------------------------------------------------------------------------------------------
static int check_sizes(const char* what, int64_t items, int32_t rank, const int32_t fs[3], const int32_t ms[3],
                       Sizes& z) {
  MPGAN_REQUIRE(fs && ms, MPGAN_ERR_SHAPE, "%s: null pointer", what);
  MPGAN_REQUIRE(items >= 1 && items <= 65535, MPGAN_ERR_SHAPE, "%s: items %lld (1 .. 65535)", what, (long long)items);
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "%s: rank %d (2 or 3)", what, (int)rank);
  for (int k = 0; k < 3; ++k) {
    z.f[k] = fs[k];
    z.m[k] = ms[k];
    MPGAN_REQUIRE(z.f[k] >= 1 && z.f[k] <= kMaxExtent && z.m[k] >= 1 && z.m[k] <= kMaxExtent, MPGAN_ERR_SHAPE,
                  "%s: axis %c: fixed extent %d, moving extent %d (each in [1, 2^22])", what, "xyz"[k], z.f[k], z.m[k]);
  }
  MPGAN_REQUIRE(rank == 3 || (z.f[2] == 1 && z.m[2] == 1), MPGAN_ERR_SHAPE, "%s: rank 2 with z extents %d, %d", what,
                z.f[2], z.m[2]);
  const double nf = (double)z.f[0] * z.f[1] * z.f[2], nm = (double)z.m[0] * z.m[1] * z.m[2];
  MPGAN_REQUIRE(nf <= (double)(1 << 27) && nm * items * 3 < 0x1p62, MPGAN_ERR_SHAPE,
                "%s: %g fixed voxels per item (at most 2^27)", what, nf);
  return 0;
}

static int make_level(const char* what, const Sizes& z, int32_t shrink, int32_t bins, Level& L, int& chunks) {
  MPGAN_REQUIRE(shrink >= 1 && shrink <= 64, MPGAN_ERR_SHAPE, "%s: shrink %d (1 .. 64)", what, (int)shrink);
  MPGAN_REQUIRE(bins >= 8 && bins <= kMaxBins, MPGAN_ERR_SHAPE, "%s: bins %d (8 .. 128)", what, (int)bins);
  L.shrink = shrink;
  L.bins = bins;
  L.sx = (z.f[0] + shrink - 1) / shrink;
  L.rows = ((z.f[1] + shrink - 1) / shrink) * ((z.f[2] + shrink - 1) / shrink);
  chunks = (int)std::min<int64_t>(kMaxChunks, ceil_div(L.rows, kRowsPerCta));
  return 0;
}

static Base make_base(const double base[24], const double center[3]) {
  Base b;
  for (int i = 0; i < 24; ++i) b.map[i] = base[i];
  for (int k = 0; k < 3; ++k) b.c[k] = center[k];
  return b;
}

static bool overlap(const void* a, size_t na, const void* b, size_t nb) {
  const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
  return a && b && x < y + nb && y < x + na;
}

// Workspace layout of the metric (bytes, each part 256-aligned): keys u32[items][4], counts u64[items],
// inside u64[items], moments u64[items][6] (these four zeroed together by mattes_prepare), lt f64[items][B][B], partial f64[items][chunks][6], grad f32[items][3][moving voxels].
struct Ws {
  unsigned* keys;
  unsigned long long *counts, *inside, *moments;
  double *lt, *partial;
  float* grad;
  size_t bytes;
};

static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

static Ws layout(void* base, int64_t items, const Sizes& z, int bins) {
  Ws w;
  char* p = (char*)base;
  size_t off = 0;
  auto take = [&](size_t n) { char* q = p ? p + off : nullptr; off += align256(n); return q; };
  w.keys = (unsigned*)take(16 * items);
  w.counts = (unsigned long long*)take(8 * items);
  w.inside = (unsigned long long*)take(8 * items);
  w.moments = (unsigned long long*)take(48 * items);
  w.lt = (double*)take(8 * (size_t)items * bins * bins);
  w.partial = (double*)take(48 * (size_t)items * kMaxChunks);
  w.grad = (float*)take(12 * (size_t)items * z.m[0] * z.m[1] * z.m[2]);
  w.bytes = off;
  return w;
}

}  // namespace reg
}  // namespace mpgan

using namespace mpgan;
using namespace mpgan::reg;

extern "C" size_t mpgan_gaussian_filter_workspace(int64_t items, const int32_t size[3]) {
  if (!size || items < 1) return 0;
  return (size_t)2 * 8 * (size_t)items * size[0] * size[1] * size[2];
}

extern "C" int mpgan_gaussian_filter(const float* in, int64_t items, int32_t rank, const int32_t size[3],
                                     const int32_t radius[3], const double* taps, float* out, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  MPGAN_REQUIRE(in && out && size && radius && taps && workspace, MPGAN_ERR_SHAPE, "gaussian_filter: null pointer");
  MPGAN_REQUIRE(items >= 1, MPGAN_ERR_SHAPE, "gaussian_filter: items %lld (at least 1)", (long long)items);
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "gaussian_filter: rank %d (2 or 3)", (int)rank);
  Taps t[3];
  int off = 0;
  for (int k = 0; k < 3; ++k) {
    MPGAN_REQUIRE(size[k] >= 1 && size[k] <= kMaxExtent, MPGAN_ERR_SHAPE, "gaussian_filter: axis %c: extent %d",
                  "xyz"[k], size[k]);
    MPGAN_REQUIRE(radius[k] >= 0 && radius[k] <= kMaxRadius, MPGAN_ERR_SHAPE,
                  "gaussian_filter: axis %c: radius %d (0 .. 64)", "xyz"[k], radius[k]);
    t[k].r = radius[k];
    for (int j = 0; j <= 2 * radius[k]; ++j) {
      t[k].w[j] = taps[off + j];
      MPGAN_REQUIRE(isfinite(t[k].w[j]), MPGAN_ERR_SHAPE, "gaussian_filter: tap %d of axis %c is not finite", j,
                    "xyz"[k]);
    }
    off += 2 * radius[k] + 1;
  }
  MPGAN_REQUIRE(rank == 3 || size[2] == 1, MPGAN_ERR_SHAPE, "gaussian_filter: rank 2 with z extent %d", size[2]);
  const double vox = (double)items * size[0] * size[1] * size[2];
  MPGAN_REQUIRE(vox < 0x1p40 && (double)items * size[1] * size[2] * ceil_div(size[0], 128) < 0x1p31, MPGAN_ERR_SHAPE,
                "gaussian_filter: tensor too large");
  const size_t need = mpgan_gaussian_filter_workspace(items, size);
  MPGAN_REQUIRE(workspace_bytes >= need, MPGAN_ERR_SHAPE, "gaussian_filter: workspace %zu bytes, need %zu",
                workspace_bytes, need);
  const int64_t n = (int64_t)vox;
  MPGAN_REQUIRE(!overlap(in, 4 * n, out, 4 * n) && !overlap(workspace, need, in, 4 * n) &&
                    !overlap(workspace, need, out, 4 * n),
                MPGAN_ERR_SHAPE, "gaussian_filter: in, out and workspace overlap");
  double* a = (double*)workspace;
  double* b = a + n;
  const cudaStream_t st = (cudaStream_t)stream;
  const int chunks = (int)ceil_div(size[0], 128);
  const int64_t rows = items * size[1] * size[2];
  launch_k(gauss_x_kernel<float>, dim3((unsigned)(rows * chunks)), dim3(128), 0, st, in, a, size[0], chunks, t[0]);
  MPGAN_CHECK_LAUNCH("gauss_x_kernel");
  const unsigned blocks = (unsigned)ceil_div(n, 128);
  const int64_t plane = (int64_t)size[0] * size[1];
  if (rank == 2) {
    launch_k(gauss_line_kernel<float>, dim3(blocks), dim3(128), 0, st, (const double*)a, out, n, (int64_t)size[0],
             size[1], t[1]);
  } else {
    launch_k(gauss_line_kernel<double>, dim3(blocks), dim3(128), 0, st, (const double*)a, b, n, (int64_t)size[0],
             size[1], t[1]);
    MPGAN_CHECK_LAUNCH("gauss_line_kernel");
    launch_k(gauss_line_kernel<float>, dim3(blocks), dim3(128), 0, st, (const double*)b, out, n, plane, size[2], t[2]);
  }
  MPGAN_CHECK_LAUNCH("gauss_line_kernel");
  return 0;
}

extern "C" int mpgan_rigid_maps(const double* params, int64_t items, int32_t rank, const double base[24],
                                const double center[3], double* maps, void* stream) {
  MPGAN_REQUIRE(params && base && center && maps, MPGAN_ERR_SHAPE, "rigid_maps: null pointer");
  MPGAN_REQUIRE(items >= 1 && items <= (1 << 30), MPGAN_ERR_SHAPE, "rigid_maps: items %lld", (long long)items);
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "rigid_maps: rank %d (2 or 3)", (int)rank);
  for (int i = 0; i < 24; ++i) MPGAN_REQUIRE(isfinite(base[i]), MPGAN_ERR_SHAPE, "rigid_maps: base[%d] not finite", i);
  launch_k(rigid_maps_kernel, dim3((unsigned)ceil_div(items, 128)), dim3(128), 0, (cudaStream_t)stream, params,
           (int)items, (int)rank, make_base(base, center), maps);
  MPGAN_CHECK_LAUNCH("rigid_maps_kernel");
  return 0;
}

extern "C" int mpgan_rigid_level(double* state, int32_t* status, int64_t items, int32_t rank, const double base[24],
                                 const double center[3], const double* initial, const double t0[3], int32_t first,
                                 double step, void* stream) {
  MPGAN_REQUIRE(state && status && base && center && t0, MPGAN_ERR_SHAPE, "rigid_level: null pointer");
  MPGAN_REQUIRE(items >= 1 && items <= 65535, MPGAN_ERR_SHAPE, "rigid_level: items %lld", (long long)items);
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "rigid_level: rank %d (2 or 3)", (int)rank);
  MPGAN_REQUIRE(step > 0 && isfinite(step), MPGAN_ERR_SHAPE, "rigid_level: step %g", step);
  launch_k(rigid_level_kernel, dim3((unsigned)ceil_div(items, 128)), dim3(128), 0, (cudaStream_t)stream, state,
           (int*)status, (int)items, (int)rank, make_base(base, center), initial, t0[0], t0[1], t0[2], (int)first,
           step);
  MPGAN_CHECK_LAUNCH("rigid_level_kernel");
  return 0;
}

extern "C" int mpgan_rigid_step(double* state, int32_t* status, int64_t items, int32_t rank, const double base[24],
                                const double center[3], double min_step, int32_t last, void* stream) {
  MPGAN_REQUIRE(state && status && base && center, MPGAN_ERR_SHAPE, "rigid_step: null pointer");
  MPGAN_REQUIRE(items >= 1 && items <= 65535, MPGAN_ERR_SHAPE, "rigid_step: items %lld", (long long)items);
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "rigid_step: rank %d (2 or 3)", (int)rank);
  MPGAN_REQUIRE(min_step > 0 && isfinite(min_step), MPGAN_ERR_SHAPE, "rigid_step: min_step %g", min_step);
  launch_k(rigid_step_kernel, dim3((unsigned)ceil_div(items, 128)), dim3(128), 0, (cudaStream_t)stream, state,
           (int*)status, (int)items, (int)rank, make_base(base, center), min_step, (int)last);
  MPGAN_CHECK_LAUNCH("rigid_step_kernel");
  return 0;
}

extern "C" size_t mpgan_mattes_workspace(int64_t items, const int32_t fixed_size[3], const int32_t moving_size[3],
                                         int32_t bins) {
  Sizes z;
  if (!fixed_size || !moving_size || items < 1 || bins < 1) return 0;
  for (int k = 0; k < 3; ++k) z.f[k] = fixed_size[k], z.m[k] = moving_size[k];
  return layout(nullptr, items, z, bins).bytes;
}

extern "C" int mpgan_mattes_prepare(const float* fixed, const float* moving, const uint8_t* mask, int64_t items,
                                    int32_t rank, const int32_t fixed_size[3], const int32_t moving_size[3],
                                    int32_t shrink, int32_t bins, const double fixed_matrix[9], double min_scale,
                                    double* state, int32_t* status, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  const char* what = "mattes_prepare";
  Sizes z;
  Level L;
  int chunks = 0;
  if (int rc = check_sizes(what, items, rank, fixed_size, moving_size, z)) return rc;
  if (int rc = make_level(what, z, shrink, bins, L, chunks)) return rc;
  MPGAN_REQUIRE(fixed && moving && state && status && workspace && fixed_matrix, MPGAN_ERR_SHAPE, "%s: null pointer",
                what);
  M9 mf;
  for (int k = 0; k < 9; ++k) {
    mf.a[k] = fixed_matrix[k];
    MPGAN_REQUIRE(isfinite(mf.a[k]), MPGAN_ERR_SHAPE, "%s: fixed_matrix[%d] = %g is not finite", what, k, mf.a[k]);
  }
  MPGAN_REQUIRE(min_scale > 0 && isfinite(min_scale), MPGAN_ERR_SHAPE, "%s: min_scale %g", what, min_scale);
  const double maxn = (double)std::max(z.f[0], std::max(z.f[1], z.f[2]));
  MPGAN_REQUIRE(maxn * maxn * z.f[0] * z.f[1] * z.f[2] < 0x1p62, MPGAN_ERR_SHAPE,
                "%s: fixed grid %d x %d x %d too elongated for the exact sample moments", what, z.f[0], z.f[1], z.f[2]);
  Ws w = layout(workspace, items, z, bins);
  MPGAN_REQUIRE(workspace_bytes >= w.bytes, MPGAN_ERR_SHAPE, "%s: workspace %zu bytes, need %zu", what,
                workspace_bytes, w.bytes);
  const cudaStream_t st = (cudaStream_t)stream;
  const int64_t nm = (int64_t)z.m[0] * z.m[1] * z.m[2];
  cudaMemsetAsync(w.keys, 0, align256(16 * items) + 2 * align256(8 * items) + align256(48 * items), st);
  MPGAN_CHECK_LAUNCH("mattes_prepare: memset");
  const int rchunks = (int)std::min<int64_t>(kMaxChunks, ceil_div(std::max<int64_t>(nm, (int64_t)L.rows * L.sx), 8 * kThreads));
  launch_k(mattes_range_kernel, dim3(rchunks, (unsigned)items, 2), dim3(kThreads), 0, st, fixed, moving, mask, z, L,
           w.keys, w.counts, w.moments);
  MPGAN_CHECK_LAUNCH("mattes_range_kernel");
  launch_k(mattes_range_finalize_kernel, dim3((unsigned)ceil_div(items, 128)), dim3(128), 0, st,
           (const unsigned*)w.keys, (const unsigned long long*)w.counts, (const unsigned long long*)w.moments,
           (int)items, (int)rank, mf, min_scale, state, (int*)status);
  MPGAN_CHECK_LAUNCH("mattes_range_finalize_kernel");
  launch_k(moving_gradient_kernel, dim3((unsigned)ceil_div(items * nm, 128)), dim3(128), 0, st, moving, z, items * nm,
           w.grad);
  MPGAN_CHECK_LAUNCH("moving_gradient_kernel");
  return 0;
}

extern "C" int mpgan_mattes_evaluate(const float* fixed, const float* moving, const uint8_t* mask, int64_t items,
                                     int32_t rank, const int32_t fixed_size[3], const int32_t moving_size[3],
                                     int32_t shrink, int32_t bins, int32_t gradient, int32_t only_running,
                                     double* state, int32_t* status, int64_t* hist, double* metric, void* workspace,
                                     size_t workspace_bytes, void* stream) {
  const char* what = "mattes_evaluate";
  Sizes z;
  Level L;
  int chunks = 0;
  if (int rc = check_sizes(what, items, rank, fixed_size, moving_size, z)) return rc;
  if (int rc = make_level(what, z, shrink, bins, L, chunks)) return rc;
  MPGAN_REQUIRE(fixed && moving && state && status && hist && metric && workspace, MPGAN_ERR_SHAPE,
                "%s: null pointer", what);
  Ws w = layout(workspace, items, z, bins);
  MPGAN_REQUIRE(workspace_bytes >= w.bytes, MPGAN_ERR_SHAPE, "%s: workspace %zu bytes, need %zu", what,
                workspace_bytes, w.bytes);
  const cudaStream_t st = (cudaStream_t)stream;
  const size_t hist_bytes = 8 * (size_t)items * bins * bins;
  const int smem_h = 8 * bins * bins;
  static bool attr = false;
  if (!attr) {
    cudaFuncSetAttribute(mattes_hist_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * kMaxBins * kMaxBins);
    cudaFuncSetAttribute(mattes_hist_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * kMaxBins * kMaxBins);
    cudaFuncSetAttribute(mattes_grad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * kMaxBins * kMaxBins);
    cudaFuncSetAttribute(mattes_grad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8 * kMaxBins * kMaxBins);
    attr = true;
  }
  cudaMemsetAsync(hist, 0, hist_bytes, st);
  cudaMemsetAsync(w.inside, 0, 8 * items, st);
  MPGAN_CHECK_LAUNCH("mattes_evaluate: memset");
  const dim3 grid(chunks, (unsigned)items);
  const int only = only_running ? 1 : 0;
  if (rank == 3)
    launch_k(mattes_hist_kernel<true>, grid, dim3(kThreads), smem_h, st, fixed, moving, mask, z, L,
             (const double*)state, (const int*)status, only, (unsigned long long*)hist, w.inside);
  else
    launch_k(mattes_hist_kernel<false>, grid, dim3(kThreads), smem_h, st, fixed, moving, mask, z, L,
             (const double*)state, (const int*)status, only, (unsigned long long*)hist, w.inside);
  MPGAN_CHECK_LAUNCH("mattes_hist_kernel");
  launch_k(mattes_finalize_kernel, dim3((unsigned)items), dim3(128), 0, st, (const unsigned long long*)hist,
           (const unsigned long long*)w.inside, (int)bins, state, (int*)status, only, metric, w.lt);
  MPGAN_CHECK_LAUNCH("mattes_finalize_kernel");
  if (!gradient) return 0;
  if (rank == 3)
    launch_k(mattes_grad_kernel<true>, grid, dim3(kThreads), smem_h, st, fixed, moving, (const float*)w.grad, mask, z,
             L, (const double*)state, (const int*)status, (const double*)w.lt, w.partial);
  else
    launch_k(mattes_grad_kernel<false>, grid, dim3(kThreads), smem_h, st, fixed, moving, (const float*)w.grad, mask,
             z, L, (const double*)state, (const int*)status, (const double*)w.lt, w.partial);
  MPGAN_CHECK_LAUNCH("mattes_grad_kernel");
  launch_k(mattes_grad_reduce_kernel, dim3((unsigned)ceil_div(items, 128)), dim3(128), 0, st,
           (const double*)w.partial, chunks, (int)items, state, (const int*)status, (int)bins);
  MPGAN_CHECK_LAUNCH("mattes_grad_reduce_kernel");
  return 0;
}
