// Intensity transforms and volume metrics on either side of the generator (SURVEY.md section 8f, rows N1 / N2):
//   * exact order statistics of an fp32 volume (np.percentile's k-th smallest values) by a two-level 16-bit radix
//     select -- MONAI ScaleIntensityRangePercentilesd(lower=1, upper=99) before training
//     (/root/reference/code/GAN/GAN_final.py:386-394) and (lower=0, upper=100) after inference
//     (/root/reference/code/GAN/inferrence.py:147-204);
//   * the affine rescale (+ clip, + np.round) with the reference's operation order in IEEE fp32 (no FMA contraction),
//     so that the rounded 0..255 volumes are bit-exact;
//   * sum |a-b| and sum (a-b)^2 in one pass (torchmetrics MeanAbsoluteError / MeanSquaredError,
//     inferrence.py:170-176, metrics.py:213-218), optionally restricted to a mask, with its voxel count.
// All of it is HBM-bound streaming / histogram work: 16-byte loads, grid-stride loops, grids sized from the SM count.
#include <cuda_fp16.h>

#include "common.cuh"

namespace mpgan {
template <> __device__ __forceinline__ __half from_f<__half>(float v) { return __float2half_rn(v); }
namespace xf {

constexpr int kThreads = 256;

// one histogram increment per distinct bin per warp: MRI volumes are ~40 % identical background voxels, and a plain
// atomicAdd per element would serialise on that one counter
__device__ __forceinline__ void hist_add(uint32_t* hist, uint32_t bin) {
  const unsigned m = __match_any_sync(__activemask(), bin);
  if ((int)(threadIdx.x & 31) == __ffs(m) - 1) atomicAdd(&hist[bin], (uint32_t)__popc(m));
}

// pass 1: histogram of the high 16 key bits (global atomics; the volume is read once)
__global__ void __launch_bounds__(kThreads) hist_hi_kernel(const float* __restrict__ x, int64_t n, uint32_t* __restrict__ hist) {
  pdl_wait();
  pdl_launch();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t n4 = n / 4;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = x4[i];
    hist_add(hist, key_of(v.x) >> 16);
    hist_add(hist, key_of(v.y) >> 16);
    hist_add(hist, key_of(v.z) >> 16);
    hist_add(hist, key_of(v.w) >> 16);
  }
  for (int64_t i = n4 * 4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    hist_add(hist, key_of(x[i]) >> 16);
}

// pass 2 / 4 (one block): locate, for every requested rank, the bin that contains it and the rank inside the bin.
// sel[r] = {bin, rank inside bin (low, high 32 bits)}.  `ranks_in` are read from sel when `chained` (second level).
__global__ void __launch_bounds__(1024) find_bin_kernel(const uint32_t* __restrict__ hist, int nbins_log2, int nr,
                                                         const int64_t* __restrict__ ranks, uint32_t* __restrict__ sel,
                                                         int chained) {
  pdl_wait();
  pdl_launch();
  __shared__ unsigned long long part[1024];
  const int nbins = 1 << nbins_log2;
  const int per = nbins / 1024;   // bins per thread (64)
  for (int r = 0; r < nr; ++r) {
    const uint32_t* h = hist + (chained ? (size_t)r * nbins : 0);
    unsigned long long want = chained ? ((unsigned long long)sel[4 * r + 1] | ((unsigned long long)sel[4 * r + 2] << 32))
                                      : (unsigned long long)ranks[r];
    unsigned long long s = 0;
    for (int j = 0; j < per; ++j) s += h[threadIdx.x * per + j];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {   // 1024-entry serial scan: negligible, and exact
      unsigned long long acc = 0;
      int t = 0;
      for (; t < 1024; ++t) {
        if (acc + part[t] > want) break;
        acc += part[t];
      }
      if (t == 1024) t = 1023;   // rank == n (cannot happen for valid ranks)
      int b = t * per;
      for (; b < t * per + per - 1; ++b) {
        if (acc + h[b] > want) break;
        acc += h[b];
      }
      const unsigned long long inside = want - acc;
      if (!chained) {
        sel[4 * r] = (uint32_t)b;
        sel[4 * r + 1] = (uint32_t)inside;
        sel[4 * r + 2] = (uint32_t)(inside >> 32);
      } else {
        sel[4 * r + 3] = (sel[4 * r] << 16) | (uint32_t)b;   // full 32-bit key of the rank-th smallest value
      }
    }
    __syncthreads();
  }
}

// pass 3: histograms of the low 16 key bits, one per requested rank, over the elements of that rank's high bin
__global__ void __launch_bounds__(kThreads) hist_lo_kernel(const float* __restrict__ x, int64_t n, int nr,
                                                           const uint32_t* __restrict__ sel, uint32_t* __restrict__ hist2) {
  pdl_wait();
  pdl_launch();
  uint32_t bins[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) bins[r] = r < nr ? sel[4 * r] : 0xffffffffu;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint32_t k = key_of(x[i]);
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if ((k >> 16) == bins[r]) hist_add(hist2 + (size_t)r * 65536, k & 0xffffu);
  }
}

// ranks 0 and n-1 (the 0 / 100 percentiles of the post-processing transform) are a plain min / max reduction
__global__ void __launch_bounds__(kThreads) minmax_key_kernel(const float* __restrict__ x, int64_t n, uint32_t* __restrict__ mm) {
  pdl_wait();
  pdl_launch();
  uint32_t lo = 0xffffffffu, hi = 0u;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t n4 = n / 4;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    const float4 v = x4[i];
    const uint32_t a = key_of(v.x), b = key_of(v.y), c = key_of(v.z), d = key_of(v.w);
    lo = min(lo, min(min(a, b), min(c, d)));
    hi = max(hi, max(max(a, b), max(c, d)));
  }
  for (int64_t i = n4 * 4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint32_t a = key_of(x[i]);
    lo = min(lo, a); hi = max(hi, a);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
  }
  if ((threadIdx.x & 31) == 0) { atomicMin(&mm[0], lo); atomicMax(&mm[1], hi); }
}

__global__ void write_minmax_kernel(const uint32_t* __restrict__ mm, const int64_t* __restrict__ ranks, int nr,
                                    float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  if ((int)threadIdx.x < nr) out[threadIdx.x] = value_of(ranks[threadIdx.x] == 0 ? mm[0] : mm[1]);
}

__global__ void write_values_kernel(const uint32_t* __restrict__ sel, int nr, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  if ((int)threadIdx.x < nr) out[threadIdx.x] = value_of(sel[4 * threadIdx.x + 3]);
}

// y = clip(((x - a_min) / (a_max - a_min)) * (b_max - b_min) + b_min)   [np.round]   -- MONAI ScaleIntensityRange
// order of operations, every step rounded to fp32 (numpy float32 array arithmetic).  a_max == a_min: x - a_min + b_min.
template <typename TO>
__global__ void __launch_bounds__(kThreads) rescale_kernel(const float* __restrict__ x, int64_t n, float a_min, float a_max,
                                                           float b_min, float b_max, int do_clip, float c_lo, float c_hi,
                                                           int do_round, TO* __restrict__ y) {
  pdl_wait();
  pdl_launch();
  const float den = __fsub_rn(a_max, a_min), span = __fsub_rn(b_max, b_min);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float v = __fsub_rn(x[i], a_min);
    if (den != 0.f) {
      v = __fdiv_rn(v, den);
      v = __fadd_rn(__fmul_rn(v, span), b_min);
    } else {
      v = __fadd_rn(v, b_min);
    }
    if (do_clip) v = fminf(fmaxf(v, c_lo), c_hi);
    if (do_round) v = rintf(v);   // round half to even, like np.round
    y[i] = from_f<TO>(v);
  }
}

// out[0] += sum |a-b|, out[1] += sum (a-b)^2; kMasked: only where mask[i] != 0 (a select, so NaN / inf outside the mask
// never reach the sums), and out[2] += the number of such voxels
template <bool kMasked>
__global__ void __launch_bounds__(kThreads) err_sums_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                            const uint8_t* __restrict__ mask, int64_t n,
                                                            double* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  constexpr int kSums = kMasked ? 3 : 2;
  __shared__ double red[kSums][kThreads / 32];
  double s1 = 0.0, s2 = 0.0, s3 = 0.0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    if constexpr (kMasked) {
      if (!mask[i]) continue;
      s3 += 1.0;
    }
    const float d = a[i] - b[i];
    s1 += (double)fabsf(d);
    s2 += (double)d * (double)d;
  }
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s1; red[1][threadIdx.x >> 5] = s2; }
  if constexpr (kMasked) {
    s3 = warp_sum(s3);
    if ((threadIdx.x & 31) == 0) red[2][threadIdx.x >> 5] = s3;
  }
  __syncthreads();
  if (threadIdx.x < kSums) {
    double t = 0.0;
    for (int i = 0; i < kThreads / 32; ++i) t += red[threadIdx.x][i];
    atomicAdd(&out[threadIdx.x], t);
  }
}

static int grid_for(int64_t n, int per_thread) {
  int64_t b = ceil_div(n, (int64_t)kThreads * per_thread);
  const int64_t cap = (int64_t)num_sms() * 8;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace xf
}  // namespace mpgan

using namespace mpgan;

extern "C" size_t mpgan_order_stats_workspace(int32_t nranks) {
  return (size_t)65536 * 4 + (size_t)nranks * 65536 * 4 + 64 * 4;   // hi histogram, lo histograms, selection records
}

extern "C" int mpgan_minmax(const float* x, int64_t n, const int64_t* ranks_dev, int32_t nranks, float* out,
                            void* workspace, size_t workspace_bytes, void* stream) {
  MPGAN_REQUIRE(x && ranks_dev && out && workspace, MPGAN_ERR_SHAPE, "minmax: null pointer");
  MPGAN_REQUIRE(n > 0, MPGAN_ERR_SHAPE, "minmax: empty volume");
  MPGAN_REQUIRE(nranks >= 1 && nranks <= 4, MPGAN_ERR_UNSUPPORTED, "minmax: 1..4 ranks per call");
  MPGAN_REQUIRE(workspace_bytes >= 8, MPGAN_ERR_SHAPE, "minmax: workspace too small");
  MPGAN_REQUIRE(((uintptr_t)x & 15) == 0, MPGAN_ERR_SHAPE, "minmax: volume not 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  uint32_t* mm = (uint32_t*)workspace;
  cudaError_t e = cudaMemsetAsync(mm, 0xff, 4, s);
  if (e == cudaSuccess) e = cudaMemsetAsync(mm + 1, 0, 4, s);
  MPGAN_REQUIRE(e == cudaSuccess, MPGAN_ERR_CUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
  launch_k(xf::minmax_key_kernel, xf::grid_for(n, 32), xf::kThreads, 0, s, x, n, mm);
  MPGAN_CHECK_LAUNCH("minmax_key_kernel");
  launch_k(xf::write_minmax_kernel, 1, 32, 0, s, (const uint32_t*)mm, ranks_dev, (int)nranks, out);
  MPGAN_CHECK_LAUNCH("write_minmax_kernel");
  return 0;
}

extern "C" int mpgan_order_stats(const float* x, int64_t n, const int64_t* ranks_dev, int32_t nranks, float* out,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  MPGAN_REQUIRE(x && ranks_dev && out && workspace, MPGAN_ERR_SHAPE, "order_stats: null pointer");
  MPGAN_REQUIRE(n > 0, MPGAN_ERR_SHAPE, "order_stats: empty volume");
  MPGAN_REQUIRE(nranks >= 1 && nranks <= 4, MPGAN_ERR_UNSUPPORTED, "order_stats: 1..4 ranks per call");
  MPGAN_REQUIRE(workspace_bytes >= mpgan_order_stats_workspace(nranks), MPGAN_ERR_SHAPE, "order_stats: workspace too small");
  MPGAN_REQUIRE(((uintptr_t)x & 15) == 0, MPGAN_ERR_SHAPE, "order_stats: volume not 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  uint32_t* hist = (uint32_t*)workspace;
  uint32_t* hist2 = hist + 65536;
  uint32_t* sel = hist2 + (size_t)nranks * 65536;
  cudaError_t e = cudaMemsetAsync(workspace, 0, mpgan_order_stats_workspace(nranks), s);
  MPGAN_REQUIRE(e == cudaSuccess, MPGAN_ERR_CUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
  launch_k(xf::hist_hi_kernel, xf::grid_for(n, 16), xf::kThreads, 0, s, x, n, hist);
  MPGAN_CHECK_LAUNCH("hist_hi_kernel");
  launch_k(xf::find_bin_kernel, 1, 1024, 0, s, (const uint32_t*)hist, 16, (int)nranks, ranks_dev, sel, 0);
  MPGAN_CHECK_LAUNCH("find_bin_kernel");
  launch_k(xf::hist_lo_kernel, xf::grid_for(n, 8), xf::kThreads, 0, s, x, n, (int)nranks, (const uint32_t*)sel, hist2);
  MPGAN_CHECK_LAUNCH("hist_lo_kernel");
  launch_k(xf::find_bin_kernel, 1, 1024, 0, s, (const uint32_t*)hist2, 16, (int)nranks, ranks_dev, sel, 1);
  MPGAN_CHECK_LAUNCH("find_bin_kernel");
  launch_k(xf::write_values_kernel, 1, 32, 0, s, (const uint32_t*)sel, (int)nranks, out);
  MPGAN_CHECK_LAUNCH("write_values_kernel");
  return 0;
}

extern "C" int mpgan_rescale_intensity(const float* x, int64_t n, float a_min, float a_max, float b_min, float b_max,
                                       int clip, float clip_lo, float clip_hi, int round_, int out_dtype, void* y,
                                       void* stream) {
  MPGAN_REQUIRE(x && y, MPGAN_ERR_SHAPE, "rescale_intensity: null pointer");
  MPGAN_REQUIRE(n >= 0, MPGAN_ERR_SHAPE, "rescale_intensity: negative size");
  MPGAN_REQUIRE(out_dtype == MPGAN_F32 || out_dtype == 2, MPGAN_ERR_UNSUPPORTED, "rescale_intensity: out dtype f32 (0) or f16 (2)");
  if (n == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const int grid = xf::grid_for(n, 8);
  if (out_dtype == MPGAN_F32)
    launch_k(xf::rescale_kernel<float>, grid, xf::kThreads, 0, s, x, n, a_min, a_max, b_min, b_max, clip, clip_lo, clip_hi,
             round_, (float*)y);
  else
    launch_k(xf::rescale_kernel<__half>, grid, xf::kThreads, 0, s, x, n, a_min, a_max, b_min, b_max, clip, clip_lo, clip_hi,
             round_, (__half*)y);
  MPGAN_CHECK_LAUNCH("rescale_kernel");
  return 0;
}

extern "C" int mpgan_err_sums(const float* a, const float* b, int64_t n, double* out2, void* stream) {
  MPGAN_REQUIRE(a && b && out2, MPGAN_ERR_SHAPE, "err_sums: null pointer");
  MPGAN_REQUIRE(n >= 0, MPGAN_ERR_SHAPE, "err_sums: negative size");
  if (n == 0) return 0;
  launch_k(xf::err_sums_kernel<false>, xf::grid_for(n, 8), xf::kThreads, 0, (cudaStream_t)stream, a, b,
           (const uint8_t*)nullptr, n, out2);
  MPGAN_CHECK_LAUNCH("err_sums_kernel");
  return 0;
}

extern "C" int mpgan_err_sums_masked(const float* a, const float* b, const uint8_t* mask, int64_t n, double* out3,
                                     void* stream) {
  MPGAN_REQUIRE(a && b && mask && out3, MPGAN_ERR_SHAPE, "err_sums_masked: null pointer");
  MPGAN_REQUIRE(n >= 0, MPGAN_ERR_SHAPE, "err_sums_masked: negative size");
  if (n == 0) return 0;
  launch_k(xf::err_sums_kernel<true>, xf::grid_for(n, 8), xf::kThreads, 0, (cudaStream_t)stream, a, b, mask, n, out3);
  MPGAN_CHECK_LAUNCH("err_sums_kernel");
  return 0;
}
