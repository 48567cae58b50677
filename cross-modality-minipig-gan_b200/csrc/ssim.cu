// Structural similarity (SSIM) of generated-vs-true volumes, scikit-image's `structural_similarity` with its defaults
// (the reference scores its generator with it: code/GAN/psnr_ssim_metric.py:88-95, SURVEY.md section 2).
//
// S = (2 ux uy + C1)(2 vxy + C2) / ((ux^2 + uy^2 + C1)(vx + vy + C2)), where ux, uy, uxx, uyy, uxy are the five moments
// x, y, x*x, y*y, x*y filtered by a separable window (the same 1-D taps along every spatial axis: uniform or Gaussian,
// the caller passes the taps) and v* = cov_norm * (u** - u* u*).  The mean SSIM is the mean of S over the interior,
// i.e. the voxels whose window lies inside the image, so no border mode enters and only that valid region is computed.
//
// One pass over the inputs, nothing but the per-item sums written to HBM: one CTA per (item, 16x32 output tile of the
// h-w plane, chunk of output planes along d).  The CTA marches along d; per input plane it stages the fp32 halo tile in
// shared memory, filters along w (fp64, products formed on the fly) and along h (fp64, two output rows per thread,
// register-blocked) and keeps the last `win` h-w-filtered planes of its own voxels in a thread-private shared-memory
// ring, from which the d filter gathers.  Every window sum accumulates in fp64 and S is evaluated in fp64: fp32 running
// sums along an axis miss a 1e-7 tolerance on the mean.  A block reduction and one fp64 atomicAdd per CTA end the
// kernel (the err_sums / BatchNorm statistics pattern).
#include "common.cuh"

namespace mpgan {
namespace ssim {

constexpr int kTW = 32;        // output columns per tile: one warp wide
constexpr int kR = 2;          // output rows per thread in the h pass
constexpr int kMaxWin = 15;
constexpr int kMaxWarps = 8;   // blockDim = (32, G), G in {8, 4, 2, 1}
constexpr size_t kSmemBudget = 226 * 1024;   // dynamic shared memory; the static part is < 1 KB

struct Taps { double t[kMaxWin]; };

__host__ __device__ inline size_t smem_bytes(int g, int win, int wd) {
  const size_t hh = (size_t)kR * g + win - 1, ww = (size_t)kTW + win - 1;
  return (size_t)wd * 5 * kR * kTW * g * sizeof(double)   // ring of h-w-filtered planes (thread-private slots)
         + 5 * hh * kTW * sizeof(double)                    // w-filtered moments of the halo rows
         + 2 * hh * ww * sizeof(float);                     // fp32 halo tile of x and y
}

// a, b: items x (d, h, w) contiguous.  wd = win for rank 3, 1 for rank 2 (no filter along d).
// kMasked: S enters out[item] only at interior voxels whose centre has mask != 0 (the windows still read every voxel),
// and cnt[item] += the number of those centres.
template <bool kMasked>
__global__ void __launch_bounds__(kTW * kMaxWarps) ssim_sums_kernel(
    const float* __restrict__ a, const float* __restrict__ b, const uint8_t* __restrict__ mask, int d, int h, int w,
    int win, int wd, const __grid_constant__ Taps taps, double c1, double c2, double cov_norm, int tiles_w, int tiles,
    int chunks, int clen, double* __restrict__ out, double* __restrict__ cnt) {
  pdl_wait();
  pdl_launch();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ double tap_s[kMaxWin], tap_d[kMaxWin], red[kMasked ? 2 : 1][kMaxWarps];
  const int g = blockDim.y, nthr = kTW * g, tx = threadIdx.x, tid = threadIdx.y * kTW + tx;
  const int th = kR * g, hh = th + win - 1, ww = kTW + win - 1;
  const int od = d - wd + 1, oh = h - win + 1, ow = w - win + 1;
  int bid = blockIdx.x;
  const int tile = bid % tiles;
  bid /= tiles;
  const int chunk = bid % chunks, item = bid / chunks;
  const int oh0 = (tile / tiles_w) * th, ow0 = (tile % tiles_w) * kTW;
  const int o_lo = chunk * clen, o_hi = min(od, o_lo + clen);

  double* ring = reinterpret_cast<double*>(smem_raw);   // [wd][5][kR][nthr]
  double* hs = ring + (size_t)wd * 5 * kR * nthr;        // [5][hh][kTW]
  float* xs = reinterpret_cast<float*>(hs + 5 * hh * kTW);   // [2][hh][ww]
  if (tid < win) {
    tap_s[tid] = taps.t[tid];
    tap_d[tid] = wd == 1 ? 1.0 : taps.t[tid];
  }
  const size_t plane = (size_t)h * w;
  const float* ai = a + (size_t)item * d * plane;
  const float* bi = b + (size_t)item * d * plane;
  const int r0 = threadIdx.y * kR;   // first of this thread's output rows in the tile
  double acc = 0.0, nacc = 0.0;

  for (int z = o_lo; z < o_hi + wd - 1; ++z) {
    // 1. halo tile of plane z (zero outside the image: those voxels only feed outputs outside the interior)
    for (int i = tid; i < hh * ww; i += nthr) {
      const int r = i / ww, c = i - r * ww;
      const int gh = oh0 + r, gw = ow0 + c;
      float va = 0.f, vb = 0.f;
      if (gh < h && gw < w) {
        const size_t off = (size_t)z * plane + (size_t)gh * w + gw;
        va = ai[off];
        vb = bi[off];
      }
      xs[i] = va;
      xs[hh * ww + i] = vb;
    }
    __syncthreads();
    // 2. filter along w: the five moments of every halo row at the tile's kTW output columns
    for (int i = tid; i < hh * kTW; i += nthr) {
      const int r = i / kTW;   // column = tx (nthr is a multiple of kTW)
      const float* px = xs + r * ww + tx;
      const float* py = px + hh * ww;
      double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0, m4 = 0.0;
      for (int k = 0; k < win; ++k) {
        const double x = px[k], y = py[k], t = tap_s[k];
        const double tx_ = t * x, ty_ = t * y;
        m0 += tx_;
        m1 += ty_;
        m2 = fma(tx_, x, m2);
        m3 = fma(ty_, y, m3);
        m4 = fma(tx_, y, m4);
      }
      hs[0 * hh * kTW + i] = m0;
      hs[1 * hh * kTW + i] = m1;
      hs[2 * hh * kTW + i] = m2;
      hs[3 * hh * kTW + i] = m3;
      hs[4 * hh * kTW + i] = m4;
    }
    __syncthreads();
    // 3. filter along h: rows r0 .. r0 + kR - 1 of the tile share win + kR - 2 of their win input rows
    double p[kR][5];
#pragma unroll
    for (int rr = 0; rr < kR; ++rr)
#pragma unroll
      for (int m = 0; m < 5; ++m) p[rr][m] = 0.0;
    for (int k = 0; k < win + kR - 1; ++k) {
      double v[5];
#pragma unroll
      for (int m = 0; m < 5; ++m) v[m] = hs[m * hh * kTW + (r0 + k) * kTW + tx];
#pragma unroll
      for (int rr = 0; rr < kR; ++rr) {
        const int kk = k - rr;
        if (kk >= 0 && kk < win) {
          const double t = tap_s[kk];
#pragma unroll
          for (int m = 0; m < 5; ++m) p[rr][m] = fma(t, v[m], p[rr][m]);
        }
      }
    }
    // 4. ring slot of plane z; once win planes are in, filter along d and evaluate S for output plane z - wd + 1
    const int slot = z % wd;
#pragma unroll
    for (int m = 0; m < 5; ++m)
#pragma unroll
      for (int rr = 0; rr < kR; ++rr) ring[((size_t)(slot * 5 + m) * kR + rr) * nthr + tid] = p[rr][m];
    if (z >= o_lo + wd - 1) {
      const int o = z - wd + 1;
      double u[kR][5];
#pragma unroll
      for (int rr = 0; rr < kR; ++rr)
#pragma unroll
        for (int m = 0; m < 5; ++m) u[rr][m] = 0.0;
      for (int k = 0; k < wd; ++k) {
        const int s = (o + k) % wd;
        const double t = tap_d[k];
#pragma unroll
        for (int m = 0; m < 5; ++m)
#pragma unroll
          for (int rr = 0; rr < kR; ++rr) u[rr][m] = fma(t, ring[((size_t)(s * 5 + m) * kR + rr) * nthr + tid], u[rr][m]);
      }
#pragma unroll
      for (int rr = 0; rr < kR; ++rr) {
        if (oh0 + r0 + rr >= oh || ow0 + tx >= ow) continue;
        if constexpr (kMasked) {
          const int half = (win - 1) / 2;
          if (!mask[(size_t)item * d * plane + (size_t)(o + (wd - 1) / 2) * plane + (size_t)(oh0 + r0 + rr + half) * w +
                    ow0 + tx + half])
            continue;
          nacc += 1.0;
        }
        // explicit roundings (no FMA contraction): with x == y every factor of the numerator equals its counterpart in
        // the denominator bit for bit, so identical images score exactly 1
        const double ux = u[rr][0], uy = u[rr][1], uxx = u[rr][2], uyy = u[rr][3], uxy = u[rr][4];
        const double uxuy = __dmul_rn(ux, uy), ux2 = __dmul_rn(ux, ux), uy2 = __dmul_rn(uy, uy);
        const double vx = __dmul_rn(cov_norm, __dsub_rn(uxx, ux2));
        const double vy = __dmul_rn(cov_norm, __dsub_rn(uyy, uy2));
        const double vxy = __dmul_rn(cov_norm, __dsub_rn(uxy, uxuy));
        const double num = __dmul_rn(__dadd_rn(__dmul_rn(2.0, uxuy), c1), __dadd_rn(__dmul_rn(2.0, vxy), c2));
        const double den = __dmul_rn(__dadd_rn(__dadd_rn(ux2, uy2), c1), __dadd_rn(__dadd_rn(vx, vy), c2));
        acc += __ddiv_rn(num, den);
      }
    }
    __syncthreads();   // xs / hs are overwritten by the next plane
  }
  acc = warp_sum(acc);
  if (tx == 0) red[0][threadIdx.y] = acc;
  if constexpr (kMasked) {
    nacc = warp_sum(nacc);
    if (tx == 0) red[1][threadIdx.y] = nacc;
  }
  __syncthreads();
  if (tid == 0) {
    double t = 0.0;
    for (int i = 0; i < g; ++i) t += red[0][i];
    atomicAdd(&out[item], t);
    if constexpr (kMasked) {
      t = 0.0;
      for (int i = 0; i < g; ++i) t += red[1][i];
      atomicAdd(&cnt[item], t);
    }
  }
}

}  // namespace ssim
}  // namespace mpgan

using namespace mpgan;

template <bool kMasked>
static int ssim_sums(const float* a, const float* b, const uint8_t* mask, int32_t rank, int32_t items, int32_t d,
                     int32_t h, int32_t w, const double* taps, int32_t win, double c1, double c2, double cov_norm,
                     double* out, double* cnt, void* stream) {
  using namespace mpgan::ssim;
  MPGAN_REQUIRE(a && b && taps && out && (!kMasked || (mask && cnt)), MPGAN_ERR_SHAPE, "ssim_sums: null pointer");
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "ssim_sums: rank %d (2 or 3)", (int)rank);
  MPGAN_REQUIRE(win >= 3 && win <= kMaxWin && (win & 1), MPGAN_ERR_UNSUPPORTED, "ssim_sums: window %d (odd, 3..%d)",
                (int)win, kMaxWin);
  MPGAN_REQUIRE(items >= 1 && h >= win && w >= win && (rank == 2 ? d == 1 : d >= win), MPGAN_ERR_SHAPE,
                "ssim_sums: items %d x (%d, %d, %d) has no interior for window %d at rank %d", (int)items, (int)d, (int)h,
                (int)w, (int)win, (int)rank);
  const int wd = rank == 3 ? win : 1;
  int g = kMaxWarps;
  while (g > 1 && smem_bytes(g, win, wd) > kSmemBudget) g >>= 1;
  const size_t smem = smem_bytes(g, win, wd);
  const int od = d - wd + 1, oh = h - win + 1, ow = w - win + 1;
  const int tiles_w = (int)ceil_div(ow, kTW), tiles = tiles_w * (int)ceil_div(oh, (int64_t)kR * g);
  // split d into chunks of output planes when (tiles x items) alone would leave SMs idle; each chunk re-reads the
  // wd - 1 planes before it, so chunks stay at least 2 (wd - 1) planes long
  int chunks = 1;
  if (wd > 1) {
    const int64_t want = ceil_div(4 * (int64_t)num_sms(), (int64_t)tiles * items);
    const int64_t cap = od / (2 * (wd - 1)) > 1 ? od / (2 * (wd - 1)) : 1;
    chunks = (int)(want < cap ? want : cap);
  }
  const int clen = (int)ceil_div(od, chunks);
  chunks = (int)ceil_div(od, clen);
  const int64_t blocks = (int64_t)tiles * chunks * items;
  MPGAN_REQUIRE(blocks <= 0x7fffffff, MPGAN_ERR_SHAPE, "ssim_sums: too many tiles");
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(ssim_sums_kernel<kMasked>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kSmemBudget);
    MPGAN_REQUIRE(e == cudaSuccess, MPGAN_ERR_CUDA, "cudaFuncSetAttribute(ssim_sums): %s", cudaGetErrorString(e));
    attr_done = true;
  }
  Taps t;
  for (int i = 0; i < kMaxWin; ++i) t.t[i] = i < win ? taps[i] : 0.0;
  launch_k(ssim_sums_kernel<kMasked>, (unsigned)blocks, dim3(kTW, g), smem, (cudaStream_t)stream, a, b, mask, (int)d,
           (int)h, (int)w, (int)win, wd, t, c1, c2, cov_norm, tiles_w, tiles, chunks, clen, out, cnt);
  MPGAN_CHECK_LAUNCH("ssim_sums_kernel");
  return 0;
}

extern "C" int mpgan_ssim_sums(const float* a, const float* b, int32_t rank, int32_t items, int32_t d, int32_t h,
                               int32_t w, const double* taps, int32_t win, double c1, double c2, double cov_norm,
                               double* out, void* stream) {
  return ssim_sums<false>(a, b, nullptr, rank, items, d, h, w, taps, win, c1, c2, cov_norm, out, nullptr, stream);
}

extern "C" int mpgan_ssim_sums_masked(const float* a, const float* b, const uint8_t* mask, int32_t rank, int32_t items,
                                      int32_t d, int32_t h, int32_t w, const double* taps, int32_t win, double c1,
                                      double c2, double cov_norm, double* out, double* count, void* stream) {
  return ssim_sums<true>(a, b, mask, rank, items, d, h, w, taps, win, c1, c2, cov_norm, out, count, stream);
}
