// Mutual information of generated-vs-true volumes from their joint histogram: the numpy/scipy computation behind
// scikit-image's normalized_mutual_information(image0, image1, bins) (np.histogramdd with autodetected ranges, then
// scipy.stats.entropy of the marginals and of the joint distribution), plus plain MI from the same histogram.
// include/mpgan.h pins the semantics.
//
// Three launches, all on the caller's stream, no host round trip:
//   1. mi_minmax_kernel: per (item, chunk) CTA, min / max of both images as order-preserving keys, atomicMin / Max
//      into the workspace (NaN and +-inf come out as non-finite extremes, which later turn the item into NaN).
//   2. mi_hist_kernel: per (item, chunk) CTA, the item's two fp32 edge tables in shared memory (explicitly rounded, no
//      FMA), a private bins x bins uint32 histogram in shared memory, and one 64-bit integer atomic per non-zero bin
//      into the item's global counts: integer sums, so the result does not depend on the CTA schedule.  A bin is
//      guessed arithmetically and corrected against the edge table, so it is np.searchsorted's bin for every value.
//      ~40 % of an MRI volume is one background value, and in a generated-vs-true pair those voxels share one joint
//      bin: each warp issues one shared-memory atomic per distinct joint bin (__match_any_sync on the key).
//   3. mi_entropy_kernel: one CTA per item, the marginals and H1, H2, H12, MI, NMI in fp64.
#include "common.cuh"

namespace mpgan {
namespace mi {

constexpr int kThreads = 512;
constexpr int kEntropyThreads = 256;   // threads [0, 128) sum rows, [128, 256) columns
constexpr int kMaxBins = 128;
constexpr int64_t kMinPerCta = 16384;  // voxels: below this the per-CTA zero / merge of bins^2 counters dominates

// The voxels of one item as a float4 body, 16-byte aligned in both images (and, kMasked, 4-byte aligned in the mask),
// and at most 6 scalars around it; every voxel is a scalar when a, b (and the mask) are not aligned alike.
struct Layout {
  int64_t head, n4, ns;   // scalars before the body, float4s in the body, scalars in all
};
template <bool kMasked>
__device__ __forceinline__ Layout layout_of(const float* a, const float* b, const uint8_t* m, int64_t n) {
  const unsigned ma = (unsigned)((uintptr_t)a & 15), mb = (unsigned)((uintptr_t)b & 15);
  Layout l;
  if (ma != mb || (ma & 3) || (kMasked && (((uintptr_t)m + (((16 - ma) & 15) >> 2)) & 3))) {
    l.head = n;
    l.n4 = 0;
  } else {
    l.head = min((int64_t)(((16 - ma) & 15) >> 2), n);
    l.n4 = (n - l.head) >> 2;
  }
  l.ns = n - 4 * l.n4;
  return l;
}

// f(x, y, ok) for the voxels of chunk `chunk` of `chunks` of one item.  Every lane of a warp makes the same calls (ok is
// false past the end and, kMasked, where the mask is 0), so f may use full-warp intrinsics.
template <bool kMasked, class F>
__device__ __forceinline__ void for_chunk(const float* __restrict__ a, const float* __restrict__ b,
                                          const uint8_t* __restrict__ m, int64_t n, int chunk, int chunks, F&& f) {
  const Layout l = layout_of<kMasked>(a, b, m, n);
  const int lane = threadIdx.x & 31;
  const int64_t w0 = (int64_t)(threadIdx.x >> 5) * 32, wstep = (int64_t)blockDim.x;
  const float4* a4 = reinterpret_cast<const float4*>(a + l.head);
  const float4* b4 = reinterpret_cast<const float4*>(b + l.head);
  const int64_t q0 = l.n4 * chunk / chunks, q1 = l.n4 * (chunk + 1) / chunks;
  for (int64_t base = q0 + w0; base < q1; base += wstep) {
    const int64_t i = base + lane;
    const bool ok = i < q1;
    float4 va = make_float4(0.f, 0.f, 0.f, 0.f), vb = va;
    uchar4 vm = make_uchar4(1, 1, 1, 1);
    if (ok) {
      va = __ldg(a4 + i);
      vb = __ldg(b4 + i);
      if constexpr (kMasked) vm = __ldg(reinterpret_cast<const uchar4*>(m + l.head) + i);
    }
    f(va.x, vb.x, ok && vm.x);
    f(va.y, vb.y, ok && vm.y);
    f(va.z, vb.z, ok && vm.z);
    f(va.w, vb.w, ok && vm.w);
  }
  const int64_t s0 = l.ns * chunk / chunks, s1 = l.ns * (chunk + 1) / chunks;
  for (int64_t base = s0 + w0; base < s1; base += wstep) {
    const int64_t s = base + lane;
    const bool ok = s < s1;
    float va = 0.f, vb = 0.f;
    bool in = true;
    if (ok) {
      const int64_t e = s < l.head ? s : s + 4 * l.n4;
      va = __ldg(a + e);
      vb = __ldg(b + e);
      if constexpr (kMasked) in = __ldg(m + e) != 0;
    }
    f(va, vb, ok && in);
  }
}

// workspace: uint32 keys, [0, 2 items) minima (image 0 items, then image 1), [2 items, 4 items) maxima; kMasked: over
// the voxels with mask != 0 only (none: the keys stay at their initial values, which read back as NaN)
template <bool kMasked>
__global__ void __launch_bounds__(kThreads) mi_minmax_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                             const uint8_t* __restrict__ mask, int64_t n, int items,
                                                             int chunks, uint32_t* __restrict__ mm) {
  pdl_wait();
  pdl_launch();
  const int item = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  uint32_t lo0 = 0xffffffffu, hi0 = 0u, lo1 = 0xffffffffu, hi1 = 0u;
  for_chunk<kMasked>(a + (int64_t)item * n, b + (int64_t)item * n, kMasked ? mask + (int64_t)item * n : nullptr, n, chunk,
                     chunks, [&](float x, float y, bool ok) {
    if (ok) {
      const uint32_t kx = key_of(x), ky = key_of(y);
      lo0 = min(lo0, kx);
      hi0 = max(hi0, kx);
      lo1 = min(lo1, ky);
      hi1 = max(hi1, ky);
    }
  });
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo0 = min(lo0, __shfl_xor_sync(0xffffffffu, lo0, o));
    hi0 = max(hi0, __shfl_xor_sync(0xffffffffu, hi0, o));
    lo1 = min(lo1, __shfl_xor_sync(0xffffffffu, lo1, o));
    hi1 = max(hi1, __shfl_xor_sync(0xffffffffu, hi1, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(&mm[item], lo0);
    atomicMin(&mm[items + item], lo1);
    atomicMax(&mm[2 * items + item], hi0);
    atomicMax(&mm[3 * items + item], hi1);
  }
}

// (lo, hi) of image m of an item after np.histogramdd's widening of an empty range; false when not finite
__device__ __forceinline__ bool range_of(const uint32_t* __restrict__ mm, int items, int item, int m, float& lo, float& hi) {
  lo = value_of(mm[m * items + item]);
  hi = value_of(mm[(2 + m) * items + item]);
  if (!(isfinite(lo) && isfinite(hi))) return false;
  if (lo == hi) {
    lo = __fsub_rn(lo, 0.5f);
    hi = __fadd_rn(hi, 0.5f);
  }
  return true;
}

// edge i of np.linspace(lo, hi, bins + 1, dtype=float32) (include/mpgan.h)
__device__ __forceinline__ float edge_of(float lo, float hi, int bins, int i) {
  if (i == bins) return hi;
  const float delta = __fsub_rn(hi, lo), step = __fdiv_rn(delta, (float)bins);
  const float y = step != 0.f ? __fmul_rn((float)i, step) : __fmul_rn(__fdiv_rn((float)i, (float)bins), delta);
  return __fadd_rn(y, lo);
}

// searchsorted(e, v, side="right") - 1, capped at bins - 1, for lo <= v <= hi: the guess (v - lo) * bins / (hi - lo) is
// within a bin or two of it; the walks make it exact against the (non-decreasing) table
__device__ __forceinline__ int bin_of(float v, const float* e, float lo, float inv, float off, int bins) {
  int b = (int)fminf(fmaxf(fmaf(v - lo, inv, off), 0.f), (float)(bins - 1));
  while (b < bins - 1 && e[b + 1] <= v) ++b;
  while (b > 0 && e[b] > v) --b;
  return b;
}

template <bool kMasked>
__global__ void __launch_bounds__(kThreads) mi_hist_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                           const uint8_t* __restrict__ mask, int64_t n, int items,
                                                           int bins, int chunks,
                                                           const uint32_t* __restrict__ mm,
                                                           unsigned long long* __restrict__ counts,
                                                           float* __restrict__ edges) {
  pdl_wait();
  pdl_launch();
  extern __shared__ uint32_t hist[];   // [bins][bins]
  __shared__ float e0[kMaxBins + 1], e1[kMaxBins + 1];
  const int item = blockIdx.x / chunks, chunk = blockIdx.x % chunks, tid = threadIdx.x;
  float lo0, hi0, lo1, hi1;
  const bool finite = range_of(mm, items, item, 0, lo0, hi0) & range_of(mm, items, item, 1, lo1, hi1);
  float* ge = edges ? edges + (size_t)item * 2 * (bins + 1) : nullptr;
  if (!finite) {   // counts stay zero; the entropy kernel writes NaN
    if (ge && chunk == 0)
      for (int i = tid; i < 2 * (bins + 1); i += blockDim.x) ge[i] = __int_as_float(0x7fc00000);
    return;
  }
  for (int i = tid; i <= bins; i += blockDim.x) {
    const float x = edge_of(lo0, hi0, bins, i), y = edge_of(lo1, hi1, bins, i);
    e0[i] = x;
    e1[i] = y;
    if (ge && chunk == 0) {
      ge[i] = x;
      ge[bins + 1 + i] = y;
    }
  }
  const int nb = bins * bins;
  for (int i = tid; i < nb; i += blockDim.x) hist[i] = 0u;
  // guess parameters (plain fp32: only the walks against the table decide the bin); an empty range after widening
  // (lo - 0.5 == lo for |lo| >= 2^24) has every edge equal and every voxel in the last bin
  const float d0 = hi0 - lo0, d1 = hi1 - lo1;
  const float inv0 = d0 > 0.f ? (float)bins / d0 : 0.f, off0 = d0 > 0.f ? 0.f : (float)(bins - 1);
  const float inv1 = d1 > 0.f ? (float)bins / d1 : 0.f, off1 = d1 > 0.f ? 0.f : (float)(bins - 1);
  __syncthreads();
  const int lane = tid & 31;
  // lanes outside the item or the mask hold the key 0xffffffff and add nothing
  for_chunk<kMasked>(a + (int64_t)item * n, b + (int64_t)item * n, kMasked ? mask + (int64_t)item * n : nullptr, n, chunk,
                     chunks, [&](float x, float y, bool ok) {
    const uint32_t key = ok ? (uint32_t)(bin_of(x, e0, lo0, inv0, off0, bins) * bins + bin_of(y, e1, lo1, inv1, off1, bins))
                            : 0xffffffffu;
    const unsigned same = __match_any_sync(0xffffffffu, key);
    if (ok && lane == __ffs(same) - 1) atomicAdd(&hist[key], (uint32_t)__popc(same));
  });
  __syncthreads();
  unsigned long long* gc = counts + (size_t)item * nb;
  for (int i = tid; i < nb; i += blockDim.x) {
    const uint32_t c = hist[i];
    if (c) atomicAdd(&gc[i], (unsigned long long)c);
  }
}

__device__ __forceinline__ double plogp(unsigned long long c, double total) {
  if (!c) return 0.0;
  const double p = (double)c / total;
  return p * log(p);
}

// out5[item] = {H1, H2, H12, MI, NMI}; sums in a fixed order, so repeated calls give the same bits.  p = count / n, or
// kMasked count / (the item's total count, the voxels in its mask)
template <bool kMasked>
__global__ void __launch_bounds__(kEntropyThreads) mi_entropy_kernel(const unsigned long long* __restrict__ counts,
                                                                     int items, int bins, int64_t n,
                                                                     const uint32_t* __restrict__ mm,
                                                                     double* __restrict__ out5) {
  pdl_wait();
  pdl_launch();
  __shared__ double red[3][kEntropyThreads / 32];
  __shared__ unsigned long long tot[kMasked ? kEntropyThreads / 32 : 1];
  const int item = blockIdx.x, tid = threadIdx.x;
  float lo, hi;
  double* o = out5 + (size_t)item * 5;
  if (!(range_of(mm, items, item, 0, lo, hi) & range_of(mm, items, item, 1, lo, hi))) {
    if (tid < 5) o[tid] = __longlong_as_double(0x7ff8000000000000ll);
    return;
  }
  const unsigned long long* c = counts + (size_t)item * bins * bins;
  double total = (double)n;
  if constexpr (kMasked) {
    unsigned long long t = 0;
    for (int k = tid; k < bins * bins; k += kEntropyThreads) t += c[k];
#pragma unroll
    for (int sh = 16; sh > 0; sh >>= 1) t += __shfl_xor_sync(0xffffffffu, t, sh);
    if ((tid & 31) == 0) tot[tid >> 5] = t;
    __syncthreads();
    t = 0;
    for (int w = 0; w < kEntropyThreads / 32; ++w) t += tot[w];
    total = (double)t;
  }
  double s1 = 0.0, s2 = 0.0, s12 = 0.0;
  if (tid < bins) {   // row tid: the marginal of image 0
    unsigned long long r = 0;
    for (int j = 0; j < bins; ++j) r += c[(size_t)tid * bins + j];
    s1 = plogp(r, total);
  } else if (tid >= kMaxBins && tid - kMaxBins < bins) {   // column tid - 128: the marginal of image 1
    unsigned long long r = 0;
    for (int i = 0; i < bins; ++i) r += c[(size_t)i * bins + tid - kMaxBins];
    s2 = plogp(r, total);
  }
  for (int k = tid; k < bins * bins; k += kEntropyThreads) s12 += plogp(c[k], total);
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  s12 = warp_sum(s12);
  if ((tid & 31) == 0) {
    red[0][tid >> 5] = s1;
    red[1][tid >> 5] = s2;
    red[2][tid >> 5] = s12;
  }
  __syncthreads();
  if (tid == 0) {
    double h[3];
    for (int m = 0; m < 3; ++m) {
      double t = 0.0;
      for (int w = 0; w < kEntropyThreads / 32; ++w) t += red[m][w];
      h[m] = -t;
    }
    o[0] = h[0];
    o[1] = h[1];
    o[2] = h[2];
    o[3] = h[0] + h[1] - h[2];
    o[4] = (h[0] + h[1]) / h[2];   // 0 / 0 = NaN for two constant images, as numpy gives
  }
}

static int chunks_for(int64_t n, int items, int ctas_per_sm) {
  const int64_t want = ceil_div((int64_t)num_sms() * ctas_per_sm, items), cap = ceil_div(n, kMinPerCta);
  return (int)(want < cap ? want : cap);
}

// ---- Otsu's threshold (include/mpgan.h): the min / max pass above, then a 1-D histogram over the same fp32 edge table
// and bin walk, then the between-class variance of every split, serially in one thread per item ----
constexpr int kOtsuMaxBins = 256;

// counts[item][bins] (zeroed by the caller) over the item's [lo, hi]; mm from mi_minmax_kernel(x, x)
__global__ void __launch_bounds__(kThreads) otsu_hist_kernel(const float* __restrict__ x, int64_t n, int items, int bins,
                                                             int chunks, const uint32_t* __restrict__ mm,
                                                             unsigned long long* __restrict__ counts) {
  pdl_wait();
  pdl_launch();
  __shared__ uint32_t hist[kOtsuMaxBins];
  __shared__ float e[kOtsuMaxBins + 1];
  const int item = blockIdx.x / chunks, chunk = blockIdx.x % chunks, tid = threadIdx.x;
  float lo, hi;
  if (!range_of(mm, items, item, 0, lo, hi)) return;   // counts stay zero; the threshold kernel writes NaN
  for (int i = tid; i <= bins; i += blockDim.x) e[i] = edge_of(lo, hi, bins, i);
  for (int i = tid; i < bins; i += blockDim.x) hist[i] = 0u;
  const float d = hi - lo, inv = d > 0.f ? (float)bins / d : 0.f, off = d > 0.f ? 0.f : (float)(bins - 1);
  __syncthreads();
  const int lane = tid & 31;
  const float* xi = x + (int64_t)item * n;
  // one image: for_chunk is given it twice, and the second load of each vector is an L1 hit
  for_chunk<false>(xi, xi, nullptr, n, chunk, chunks, [&](float v, float, bool ok) {
    const uint32_t key = ok ? (uint32_t)bin_of(v, e, lo, inv, off, bins) : 0xffffffffu;
    const unsigned same = __match_any_sync(0xffffffffu, key);
    if (ok && lane == __ffs(same) - 1) atomicAdd(&hist[key], (uint32_t)__popc(same));
  });
  __syncthreads();
  unsigned long long* gc = counts + (size_t)item * bins;
  for (int i = tid; i < bins; i += blockDim.x)
    if (hist[i]) atomicAdd(&gc[i], (unsigned long long)hist[i]);
}

// thr[item]: the centre of the first split of largest between-class variance, every operation rounded (no FMA) in the
// order include/mpgan.h pins; NaN for a non-finite extreme, the value itself for a constant item
__global__ void __launch_bounds__(kOtsuMaxBins) otsu_threshold_kernel(const unsigned long long* __restrict__ counts,
                                                                      int items, int bins,
                                                                      const uint32_t* __restrict__ mm,
                                                                      float* __restrict__ thr) {
  pdl_wait();
  pdl_launch();
  __shared__ float c[kOtsuMaxBins];
  __shared__ long long w2[kOtsuMaxBins];
  __shared__ double mean2[kOtsuMaxBins];
  const int item = blockIdx.x, tid = threadIdx.x;
  const float lo = value_of(mm[item]), hi = value_of(mm[2 * items + item]);
  if (!(isfinite(lo) && isfinite(hi)) || lo == hi) {
    if (tid == 0) thr[item] = lo == hi ? lo : __int_as_float(0x7fc00000);
    return;
  }
  if (tid < bins) c[tid] = __fdiv_rn(__fadd_rn(edge_of(lo, hi, bins, tid), edge_of(lo, hi, bins, tid + 1)), 2.f);
  __syncthreads();
  if (tid != 0) return;
  const unsigned long long* h = counts + (size_t)item * bins;
  long long w = 0;
  double s = 0.0;
  for (int i = bins - 1; i >= 1; --i) {   // the class above split i - 1: weight and mean from the top
    w += (long long)h[i];
    s = __dadd_rn(s, __dmul_rn((double)h[i], (double)c[i]));
    w2[i] = w;
    mean2[i] = __ddiv_rn(s, (double)w);
  }
  w = 0;
  s = 0.0;
  double best = -1.0;
  int idx = 0;
  for (int i = 0; i < bins - 1; ++i) {   // a NaN variance (an empty lower class) wins, as in np.argmax
    w += (long long)h[i];
    s = __dadd_rn(s, __dmul_rn((double)h[i], (double)c[i]));
    const double dm = __dsub_rn(__ddiv_rn(s, (double)w), mean2[i + 1]);
    const double v = __dmul_rn((double)(w * w2[i + 1]), __dmul_rn(dm, dm));
    if (v != v) {
      idx = i;
      break;
    }
    if (v > best) {
      best = v;
      idx = i;
    }
  }
  thr[item] = c[idx];
}

// mask[item][i] = x[item][i] > thr[item] (false for NaN on either side)
__global__ void __launch_bounds__(kThreads) threshold_mask_kernel(const float* __restrict__ x,
                                                                  const float* __restrict__ thr, int64_t n, int chunks,
                                                                  uint8_t* __restrict__ mask) {
  pdl_wait();
  pdl_launch();
  const int item = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const float t = thr[item];
  const float* xi = x + (int64_t)item * n;
  uint8_t* mi = mask + (int64_t)item * n;
  const int64_t q1 = n * (chunk + 1) / chunks;
  for (int64_t i = n * chunk / chunks + threadIdx.x; i < q1; i += blockDim.x) mi[i] = __ldg(xi + i) > t;
}

}  // namespace mi
}  // namespace mpgan

using namespace mpgan;

extern "C" size_t mpgan_mutual_info_workspace(int32_t items) { return items > 0 ? (size_t)items * 4 * sizeof(uint32_t) : 0; }

template <bool kMasked>
static int mutual_info(const float* a, const float* b, const uint8_t* mask, int32_t items, int64_t n, int32_t bins,
                       int64_t* counts, float* edges, double* out5, void* workspace, size_t workspace_bytes,
                       void* stream) {
  using namespace mpgan::mi;
  MPGAN_REQUIRE(a && b && counts && out5 && workspace && (!kMasked || mask), MPGAN_ERR_SHAPE,
                "mutual_info: null pointer");
  MPGAN_REQUIRE(items >= 1, MPGAN_ERR_SHAPE, "mutual_info: items %d (>= 1)", (int)items);
  MPGAN_REQUIRE(n >= 1 && n <= 0x7fffffff, MPGAN_ERR_SHAPE, "mutual_info: %lld voxels per item (1 .. 2^31 - 1)",
                (long long)n);
  MPGAN_REQUIRE(bins >= 2 && bins <= kMaxBins, MPGAN_ERR_SHAPE, "mutual_info: bins %d (2 .. %d)", (int)bins, kMaxBins);
  MPGAN_REQUIRE(workspace_bytes >= mpgan_mutual_info_workspace(items), MPGAN_ERR_SHAPE, "mutual_info: workspace too small");
  const size_t smem = (size_t)bins * bins * sizeof(uint32_t);
  const int hist_per_sm = (int)(200 * 1024 / smem) < 2048 / kThreads ? (int)(200 * 1024 / smem) : 2048 / kThreads;
  const int c_mm = chunks_for(n, items, 2048 / kThreads), c_hist = chunks_for(n, items, hist_per_sm);
  const int64_t g_mm = (int64_t)items * c_mm, g_hist = (int64_t)items * c_hist;
  MPGAN_REQUIRE(g_mm <= 0x7fffffff && g_hist <= 0x7fffffff, MPGAN_ERR_SHAPE, "mutual_info: too many items");
  cudaStream_t s = (cudaStream_t)stream;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(mi_hist_kernel<kMasked>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         kMaxBins * kMaxBins * (int)sizeof(uint32_t));
    MPGAN_REQUIRE(e == cudaSuccess, MPGAN_ERR_CUDA, "cudaFuncSetAttribute(mi_hist): %s", cudaGetErrorString(e));
    attr_done = true;
  }
  uint32_t* mm = (uint32_t*)workspace;
  cudaError_t e = cudaMemsetAsync(mm, 0xff, (size_t)items * 2 * sizeof(uint32_t), s);
  if (e == cudaSuccess) e = cudaMemsetAsync(mm + 2 * (size_t)items, 0, (size_t)items * 2 * sizeof(uint32_t), s);
  if (e == cudaSuccess) e = cudaMemsetAsync(counts, 0, (size_t)items * bins * bins * sizeof(int64_t), s);
  MPGAN_REQUIRE(e == cudaSuccess, MPGAN_ERR_CUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
  launch_k(mi_minmax_kernel<kMasked>, (unsigned)g_mm, kThreads, 0, s, a, b, mask, n, (int)items, c_mm, mm);
  MPGAN_CHECK_LAUNCH("mi_minmax_kernel");
  launch_k(mi_hist_kernel<kMasked>, (unsigned)g_hist, kThreads, smem, s, a, b, mask, n, (int)items, (int)bins, c_hist,
           (const uint32_t*)mm, (unsigned long long*)counts, edges);
  MPGAN_CHECK_LAUNCH("mi_hist_kernel");
  launch_k(mi_entropy_kernel<kMasked>, (unsigned)items, kEntropyThreads, 0, s, (const unsigned long long*)counts,
           (int)items, (int)bins, n, (const uint32_t*)mm, out5);
  MPGAN_CHECK_LAUNCH("mi_entropy_kernel");
  return 0;
}

extern "C" int mpgan_mutual_info(const float* a, const float* b, int32_t items, int64_t n, int32_t bins, int64_t* counts,
                                 float* edges, double* out5, void* workspace, size_t workspace_bytes, void* stream) {
  return mutual_info<false>(a, b, nullptr, items, n, bins, counts, edges, out5, workspace, workspace_bytes, stream);
}

extern "C" int mpgan_mutual_info_masked(const float* a, const float* b, const uint8_t* mask, int32_t items, int64_t n,
                                        int32_t bins, int64_t* counts, float* edges, double* out5, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  return mutual_info<true>(a, b, mask, items, n, bins, counts, edges, out5, workspace, workspace_bytes, stream);
}

extern "C" size_t mpgan_otsu_threshold_workspace(int32_t items, int32_t bins) {
  return items > 0 && bins > 0 ? (size_t)items * 4 * sizeof(uint32_t) + (size_t)items * bins * sizeof(int64_t) : 0;
}

extern "C" int mpgan_otsu_threshold(const float* x, int32_t items, int64_t n, int32_t bins, float* thr, void* workspace,
                                    size_t workspace_bytes, void* stream) {
  using namespace mpgan::mi;
  MPGAN_REQUIRE(x && thr && workspace, MPGAN_ERR_SHAPE, "otsu_threshold: null pointer");
  MPGAN_REQUIRE(items >= 1, MPGAN_ERR_SHAPE, "otsu_threshold: items %d (>= 1)", (int)items);
  MPGAN_REQUIRE(n >= 1 && n <= 0x7fffffff, MPGAN_ERR_SHAPE, "otsu_threshold: %lld voxels per item (1 .. 2^31 - 1)",
                (long long)n);
  MPGAN_REQUIRE(bins >= 2 && bins <= kOtsuMaxBins, MPGAN_ERR_SHAPE, "otsu_threshold: bins %d (2 .. %d)", (int)bins,
                kOtsuMaxBins);
  MPGAN_REQUIRE(workspace_bytes >= mpgan_otsu_threshold_workspace(items, bins), MPGAN_ERR_SHAPE,
                "otsu_threshold: workspace too small");
  const int chunks = chunks_for(n, items, 2048 / kThreads);
  MPGAN_REQUIRE((int64_t)items * chunks <= 0x7fffffff, MPGAN_ERR_SHAPE, "otsu_threshold: too many items");
  cudaStream_t s = (cudaStream_t)stream;
  uint32_t* mm = (uint32_t*)workspace;
  unsigned long long* counts = (unsigned long long*)(mm + 4 * (size_t)items);
  cudaError_t e = cudaMemsetAsync(mm, 0xff, (size_t)items * 2 * sizeof(uint32_t), s);
  if (e == cudaSuccess) e = cudaMemsetAsync(mm + 2 * (size_t)items, 0, (size_t)items * 2 * sizeof(uint32_t), s);
  if (e == cudaSuccess) e = cudaMemsetAsync(counts, 0, (size_t)items * bins * sizeof(int64_t), s);
  MPGAN_REQUIRE(e == cudaSuccess, MPGAN_ERR_CUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
  launch_k(mi_minmax_kernel<false>, (unsigned)(items * chunks), kThreads, 0, s, x, x, (const uint8_t*)nullptr, n,
           (int)items, chunks, mm);
  MPGAN_CHECK_LAUNCH("mi_minmax_kernel");
  launch_k(otsu_hist_kernel, (unsigned)(items * chunks), kThreads, 0, s, x, n, (int)items, (int)bins, chunks,
           (const uint32_t*)mm, counts);
  MPGAN_CHECK_LAUNCH("otsu_hist_kernel");
  launch_k(otsu_threshold_kernel, (unsigned)items, kOtsuMaxBins, 0, s, (const unsigned long long*)counts, (int)items,
           (int)bins, (const uint32_t*)mm, thr);
  MPGAN_CHECK_LAUNCH("otsu_threshold_kernel");
  return 0;
}

extern "C" int mpgan_threshold_mask(const float* x, const float* thr, int32_t items, int64_t n, uint8_t* mask,
                                    void* stream) {
  using namespace mpgan::mi;
  MPGAN_REQUIRE(x && thr && mask, MPGAN_ERR_SHAPE, "threshold_mask: null pointer");
  MPGAN_REQUIRE(items >= 1, MPGAN_ERR_SHAPE, "threshold_mask: items %d (>= 1)", (int)items);
  MPGAN_REQUIRE(n >= 1 && n <= 0x7fffffff, MPGAN_ERR_SHAPE, "threshold_mask: %lld voxels per item (1 .. 2^31 - 1)",
                (long long)n);
  const int chunks = chunks_for(n, items, 2048 / kThreads);
  MPGAN_REQUIRE((int64_t)items * chunks <= 0x7fffffff, MPGAN_ERR_SHAPE, "threshold_mask: too many items");
  launch_k(threshold_mask_kernel, (unsigned)(items * chunks), kThreads, 0, (cudaStream_t)stream, x, thr, n, chunks, mask);
  MPGAN_CHECK_LAUNCH("threshold_mask_kernel");
  return 0;
}
