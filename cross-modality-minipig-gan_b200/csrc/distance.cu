// Exact Euclidean distance transform of masks (scipy.ndimage.distance_transform_edt) and the agreement of two masks:
// Dice, Jaccard, Hausdorff distance, its percentile and the average surface distances (MONAI's definitions over
// get_mask_edges surfaces).  include/mpgan.h pins the semantics.
//
// The transform is separable and exact, one launch per spatial axis (a fixed launch count, so it can be captured in a
// CUDA graph).  Squared distances are carried in fp64:
//   1. edt_rows_kernel: one warp per row of the contiguous axis (x).  A right-to-left warp scan writes the nearest "out"
//      voxel at or after x into the int32 workspace, a left-to-right scan reads it back and writes
//      f = (min(x - left, right - x) * s_x)^2, or +inf when the row has no "out" voxel.
//   2. edt_cols_kernel, once per remaining axis (y, then z): one thread per column, adjacent threads on adjacent
//      columns, so every step of the column loops reads and writes 32 consecutive fp64 values per warp.  It takes the
//      lower envelope of the parabolas f(i) + ((j - i) s)^2 (Felzenszwalb and Huttenlocher 2012) over the finite f(i);
//      +inf values never enter the envelope, so a column without a finite value stays +inf.  The envelope's vertices and
//      their f live in a workspace laid out like the image (vertex k of a column where voxel k of the column would
//      be), and f is overwritten in place.  The last pass writes sqrt(f).
// Intersections are formed as (a + b) / 2 + (f_b - f_a) / (2 s^2 (b - a)): its error is relative to the values near
// the intersection rather than to the squared coordinates.  At unit spacing every operand is an integer and distinct
// intersections differ by at least 1 / (4 L^2) for columns of length L, more than their rounding error while
// L <= 4096, so envelopes, and with them the squared distances, are exact.
//
// mask_agreement erodes both masks with mpgan_binary_morphology (the surfaces are m & ~erosion(m)), takes the
// transform of the complement of each surface (the "out" test of pass 1 reads the mask and its erosion), then:
//   agree_reduce_kernel  one pass over both masks, both erosions and (at surface voxels) both distance maps: per-CTA
//                        int64 counts, fp64 sums and maxima, and a one-byte surface code per voxel;
//   agree_combine_kernel one CTA per item adds the CTA partials in a fixed order and sets up the percentile selections
//                        from the device-side surface counts;
//   agree_hist_kernel /  8 levels of an 8-bit radix select over the 64-bit patterns of the surface distances
//   agree_select_kernel  (non-negative doubles order like their bit patterns; +inf last);
//   agree_final_kernel   one CTA per item: numpy's percentile arithmetic and the six results.
// No float atomics anywhere: every sum has a fixed order, so results are bit-identical run to run and independent of
// the other items of a batch.
#include <math.h>

#include "common.cuh"

namespace mpgan {
namespace dist {

constexpr int kRowWarps = 8;           // edt_rows_kernel: rows per CTA, one warp each
constexpr int kColThreads = 64;        // edt_cols_kernel: columns per CTA (latency-bound loops: spread over the SMs)
constexpr int kThreads = 256;          // agreement kernels
constexpr int kPer = 16;               // voxels per thread of the reduction
constexpr int kChunk = kThreads * kPer;
constexpr int kHistPer = 64;           // voxels per thread of a histogram pass
constexpr int kHistChunk = kThreads * kHistPer;
constexpr int kSel = 4;                // selections per item: P->T lower / upper rank, T->P lower / upper rank
constexpr int kBins = 256;
constexpr int kLevels = 8;             // 8-bit digits of a 64-bit key
constexpr int kNone = 0x7fffffff;

// "out" voxels of pass 1: mask == 0, or (kSurface) the surface m & ~erosion(m), whose complement is transformed.
template <bool kSurface>
__device__ __forceinline__ bool is_out(const uint8_t* __restrict__ mask, const uint8_t* __restrict__ eroded, int64_t g) {
  if constexpr (kSurface) return __ldg(mask + g) != 0 && __ldg(eroded + g) == 0;
  else return __ldg(mask + g) == 0;
}

template <bool kSurface>
__global__ void __launch_bounds__(kRowWarps * 32) edt_rows_kernel(const uint8_t* __restrict__ mask,
                                                                  const uint8_t* __restrict__ eroded, int64_t rows,
                                                                  int w, double s, int* __restrict__ right,
                                                                  double* __restrict__ f) {
  pdl_wait();
  pdl_launch();
  const int64_t row = (int64_t)blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int64_t base = row * w;
  int carry = kNone;   // nearest "out" voxel right of the chunk
  for (int64_t c0 = (int64_t)(w - 1) & ~(int64_t)31; c0 >= 0; c0 -= 32) {
    const int64_t x = c0 + lane;
    int r = x < w && is_out<kSurface>(mask, eroded, base + x) ? (int)x : kNone;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_down_sync(0xffffffffu, r, o);
      if (lane + o < 32) r = min(r, v);
    }
    r = min(r, carry);
    carry = __shfl_sync(0xffffffffu, r, 0);
    if (x < w) right[base + x] = r;
  }
  carry = -1;          // nearest "out" voxel left of the chunk
  for (int64_t c0 = 0; c0 < w; c0 += 32) {
    const int64_t x = c0 + lane;
    const int r = x < w ? right[base + x] : kNone;   // this lane wrote it: no synchronisation needed
    int l = r == x ? (int)x : -1;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, l, o);
      if (lane >= o) l = max(l, v);
    }
    l = max(l, carry);
    carry = __shfl_sync(0xffffffffu, l, 31);
    if (x < w) {
      double v = __longlong_as_double(0x7ff0000000000000ll);
      if (l >= 0 || r != kNone) {
        const int64_t dl = l >= 0 ? x - l : kNone, dr = r != kNone ? r - x : kNone;
        const double t = __dmul_rn((double)min(dl, dr), s);
        v = __dmul_rn(t, t);
      }
      f[base + x] = v;
    }
  }
}

// The intersection of the parabolas of vertices a < b.
__device__ __forceinline__ double sep(int a, double fa, int b, double fb, double two_s2) {
  return __dadd_rn(__dmul_rn((double)(a + b), 0.5), __ddiv_rn(__dsub_rn(fb, fa), __dmul_rn(two_s2, (double)(b - a))));
}

__global__ void __launch_bounds__(kColThreads) edt_cols_kernel(int64_t cols, int len, int64_t stride, double s,
                                                               int last, double* __restrict__ f,
                                                               int* __restrict__ env_v, double* __restrict__ env_f) {
  pdl_wait();
  pdl_launch();
  const int64_t c = (int64_t)blockIdx.x * kColThreads + threadIdx.x;
  if (c >= cols) return;
  const int64_t base = (c / stride) * len * stride + c % stride;
  const double inf = __longlong_as_double(0x7ff0000000000000ll);
  const double two_s2 = __dmul_rn(2.0, __dmul_rn(s, s));
  // lower envelope: vertices env[0..k]; the top vertex, its f and its left boundary in registers
  int k = -1, tv = 0;
  double tf = 0.0, tz = -inf;
  for (int q = 0; q < len; ++q) {
    const double fq = f[base + (int64_t)q * stride];
    if (fq == inf) continue;
    while (k > 0 && sep(tv, tf, q, fq, two_s2) <= tz) {
      --k;
      tv = env_v[base + (int64_t)k * stride];
      tf = env_f[base + (int64_t)k * stride];
      if (k > 0) {
        const int64_t p = base + (int64_t)(k - 1) * stride;
        tz = sep(env_v[p], env_f[p], tv, tf, two_s2);
      } else {
        tz = -inf;
      }
    }
    if (k >= 0) tz = sep(tv, tf, q, fq, two_s2);
    ++k;
    tv = q;
    tf = fq;
    env_v[base + (int64_t)k * stride] = q;
    env_f[base + (int64_t)k * stride] = fq;
  }
  if (k < 0) {   // no finite value in the column
    for (int j = 0; j < len; ++j) f[base + (int64_t)j * stride] = inf;
    return;
  }
  const int top = k;
  k = 0;
  int v = env_v[base];
  double fv = env_f[base];
  double znext = inf;   // right boundary of vertex k: the same sep() the construction computed, so the same bits
  if (top > 0) znext = sep(v, fv, env_v[base + stride], env_f[base + stride], two_s2);
  for (int j = 0; j < len; ++j) {
    while (znext < (double)j) {
      ++k;
      v = env_v[base + (int64_t)k * stride];
      fv = env_f[base + (int64_t)k * stride];
      znext = inf;
      if (k < top) {
        const int64_t p = base + (int64_t)(k + 1) * stride;
        znext = sep(v, fv, env_v[p], env_f[p], two_s2);
      }
    }
    const double t = __dmul_rn((double)(j - v), s);
    const double d2 = __dadd_rn(fv, __dmul_rn(t, t));
    f[base + (int64_t)j * stride] = last ? __dsqrt_rn(d2) : d2;
  }
}

// ---- agreement ----
struct Partial {
  long long cnt[5];     // |P|, |T|, |P & T|, |surface P|, |surface T|
  double sum[2], mx[2]; // sum and max of D(P->T), D(T->P)
};
struct Stats {
  long long cnt[5];
  double sum[2], mx[2];
};
struct Sel {
  unsigned long long prefix;   // the selected key's digits found so far
  long long rank;              // the rank inside the values that share the prefix; -1: nothing to select
};

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Per CTA of kChunk voxels of one item: counts, and sum / max of each direction's surface distances.  code (the
// erosion of P on entry) becomes bit 0 = surface of P, bit 1 = surface of T.
__global__ void __launch_bounds__(kThreads) agree_reduce_kernel(const uint8_t* __restrict__ pm,
                                                                const uint8_t* __restrict__ tm,
                                                                uint8_t* __restrict__ code,
                                                                const uint8_t* __restrict__ te,
                                                                const double* __restrict__ dist_t,
                                                                const double* __restrict__ dist_p, int64_t n,
                                                                int chunks, Partial* __restrict__ part) {
  __shared__ Partial red[kThreads / 32];
  pdl_wait();
  pdl_launch();
  const int64_t item = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const int64_t g0 = item * n + chunk * kChunk;
  const int lim = (int)min((int64_t)kChunk, n - chunk * kChunk);
  int cnt[5] = {0, 0, 0, 0, 0};
  double sum[2] = {0.0, 0.0}, mx[2] = {0.0, 0.0};
#pragma unroll 4
  for (int k = 0; k < kPer; ++k) {
    const int off = k * kThreads + threadIdx.x;
    if (off >= lim) break;
    const int64_t g = g0 + off;
    const bool p = pm[g] != 0, t = tm[g] != 0;
    const bool sp = p && code[g] == 0, st = t && te[g] == 0;
    cnt[0] += p;
    cnt[1] += t;
    cnt[2] += p && t;
    cnt[3] += sp;
    cnt[4] += st;
    if (sp) {
      const double d = dist_t[g];
      sum[0] = __dadd_rn(sum[0], d);
      mx[0] = fmax(mx[0], d);
    }
    if (st) {
      const double d = dist_p[g];
      sum[1] = __dadd_rn(sum[1], d);
      mx[1] = fmax(mx[1], d);
    }
    code[g] = (uint8_t)(sp | (st << 1));
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long c[5];
#pragma unroll
  for (int i = 0; i < 5; ++i) c[i] = (long long)__reduce_add_sync(0xffffffffu, (unsigned)cnt[i]);
  double s0 = warp_sum(sum[0]), s1 = warp_sum(sum[1]), m0 = warp_max(mx[0]), m1 = warp_max(mx[1]);
  if (lane == 0) {
    for (int i = 0; i < 5; ++i) red[warp].cnt[i] = c[i];
    red[warp].sum[0] = s0;
    red[warp].sum[1] = s1;
    red[warp].mx[0] = m0;
    red[warp].mx[1] = m1;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    Partial o = red[0];
    for (int w = 1; w < kThreads / 32; ++w) {
      for (int i = 0; i < 5; ++i) o.cnt[i] += red[w].cnt[i];
      for (int i = 0; i < 2; ++i) {
        o.sum[i] = __dadd_rn(o.sum[i], red[w].sum[i]);
        o.mx[i] = fmax(o.mx[i], red[w].mx[i]);
      }
    }
    part[blockIdx.x] = o;
  }
}

// np.percentile's (numpy 2.x, method "linear") neighbouring ranks lo <= hi and weight t of n sorted values.  numpy's
// linear method forms its virtual index as (n - 1) q, not as the general n q + (alpha + q (1 - alpha - beta)) - 1 of
// the other methods, which rounds differently.
__device__ __forceinline__ void percentile_ranks(long long n, double q, long long* lo, long long* hi, double* t) {
  const double v = __dmul_rn((double)(n - 1), q);
  const double fl = floor(v);
  if (v >= (double)(n - 1)) {
    *lo = *hi = n - 1;
  } else if (v < 0.0) {
    *lo = *hi = 0;
  } else {
    *lo = (long long)fl;
    *hi = *lo + 1;
  }
  *t = __dsub_rn(v, fl);
}

// One CTA per item: the CTA partials added in a fixed order (thread j takes chunks j, j + kThreads, ...), and the four
// selections set up from the surface counts.
__global__ void __launch_bounds__(kThreads) agree_combine_kernel(const Partial* __restrict__ part, int chunks, double q,
                                                                 Stats* __restrict__ stats, Sel* __restrict__ sel) {
  __shared__ Partial red[kThreads / 32];
  pdl_wait();
  pdl_launch();
  const Partial* p = part + (int64_t)blockIdx.x * chunks;
  long long c[5] = {0, 0, 0, 0, 0};
  double sum[2] = {0.0, 0.0}, mx[2] = {0.0, 0.0};
  for (int j = threadIdx.x; j < chunks; j += kThreads) {
    for (int i = 0; i < 5; ++i) c[i] += p[j].cnt[i];
    for (int i = 0; i < 2; ++i) {
      sum[i] = __dadd_rn(sum[i], p[j].sum[i]);
      mx[i] = fmax(mx[i], p[j].mx[i]);
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = 0; i < 5; ++i) c[i] = warp_sum_ll(c[i]);
  for (int i = 0; i < 2; ++i) {
    sum[i] = warp_sum(sum[i]);
    mx[i] = warp_max(mx[i]);
  }
  if (lane == 0) {
    for (int i = 0; i < 5; ++i) red[warp].cnt[i] = c[i];
    for (int i = 0; i < 2; ++i) {
      red[warp].sum[i] = sum[i];
      red[warp].mx[i] = mx[i];
    }
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  Stats st;
  for (int i = 0; i < 5; ++i) st.cnt[i] = 0;
  for (int i = 0; i < 2; ++i) st.sum[i] = st.mx[i] = 0.0;
  for (int w = 0; w < kThreads / 32; ++w) {
    for (int i = 0; i < 5; ++i) st.cnt[i] += red[w].cnt[i];
    for (int i = 0; i < 2; ++i) {
      st.sum[i] = __dadd_rn(st.sum[i], red[w].sum[i]);
      st.mx[i] = fmax(st.mx[i], red[w].mx[i]);
    }
  }
  stats[blockIdx.x] = st;
  for (int dir = 0; dir < 2; ++dir) {
    const long long m = st.cnt[3 + dir];
    long long lo = -1, hi = -1;
    double t = 0.0;
    if (m > 0) percentile_ranks(m, q, &lo, &hi, &t);
    sel[blockIdx.x * kSel + 2 * dir] = Sel{0ull, lo};
    sel[blockIdx.x * kSel + 2 * dir + 1] = Sel{0ull, hi};
  }
}

// One radix level: per item and selection, the histogram of digit `level` (bits 63 - 8 level .. 56 - 8 level) of the
// keys of the selection's direction that share its prefix.  Shared-memory counts, added to the item's global
// histogram with integer atomics (exact in any order).
__global__ void __launch_bounds__(kThreads) agree_hist_kernel(const uint8_t* __restrict__ code,
                                                              const double* __restrict__ dist_t,
                                                              const double* __restrict__ dist_p, int64_t n,
                                                              int chunks, int level, const Sel* __restrict__ sel,
                                                              unsigned* __restrict__ hist) {
  __shared__ unsigned h[kSel * kBins];
  pdl_wait();
  pdl_launch();
  const int64_t item = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  for (int i = threadIdx.x; i < kSel * kBins; i += kThreads) h[i] = 0;
  unsigned long long pre[kSel];
  bool on[kSel];
#pragma unroll
  for (int s = 0; s < kSel; ++s) {
    const Sel x = sel[item * kSel + s];
    pre[s] = x.prefix;
    on[s] = x.rank >= 0;
  }
  __syncthreads();
  const int shift = 56 - 8 * level;
  const unsigned long long known = level ? ~0ull << (shift + 8) : 0ull;
  const int64_t g0 = item * n + chunk * kHistChunk;
  const int lim = (int)min((int64_t)kHistChunk, n - chunk * kHistChunk);
  for (int off = threadIdx.x; off < lim; off += kThreads) {
    const int64_t g = g0 + off;
    const unsigned cd = code[g];
    if (!cd) continue;
#pragma unroll
    for (int dir = 0; dir < 2; ++dir) {
      if (!(cd & (1u << dir))) continue;
      const unsigned long long key = (unsigned long long)__double_as_longlong(dir ? dist_p[g] : dist_t[g]);
      const unsigned digit = (unsigned)(key >> shift) & (kBins - 1);
#pragma unroll
      for (int s = 2 * dir; s < 2 * dir + 2; ++s)
        if (on[s] && ((key ^ pre[s]) & known) == 0) atomicAdd(&h[s * kBins + digit], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kSel * kBins; i += kThreads)
    if (h[i]) atomicAdd(&hist[item * kSel * kBins + i], h[i]);
}

// One CTA per item: each selection moves into the bin that holds its rank; the histograms are zeroed for the next level.
__global__ void __launch_bounds__(kThreads) agree_select_kernel(int level, Sel* __restrict__ sel,
                                                                unsigned* __restrict__ hist) {
  pdl_wait();
  pdl_launch();
  unsigned* h = hist + (int64_t)blockIdx.x * kSel * kBins;
  if (threadIdx.x < kSel) {
    Sel& x = sel[blockIdx.x * kSel + threadIdx.x];
    if (x.rank >= 0) {
      const unsigned* hs = h + threadIdx.x * kBins;
      long long below = 0;
      int b = 0;
      for (; b < kBins - 1 && below + hs[b] <= x.rank; ++b) below += hs[b];
      x.prefix |= (unsigned long long)b << (56 - 8 * level);
      x.rank -= below;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kSel * kBins; i += kThreads) h[i] = 0;
}

__device__ __forceinline__ double lerp(double a, double b, double t) {   // numpy's _lerp
  const double diff = __dsub_rn(b, a);
  return t >= 0.5 ? __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, t))) : __dadd_rn(a, __dmul_rn(diff, t));
}

// One CTA per item (thread 0): out6 = dice, jaccard, hausdorff, hausdorff_percentile, average_surface_distance,
// symmetric_surface_distance.
__global__ void agree_final_kernel(const Stats* __restrict__ stats, const Sel* __restrict__ sel, double q,
                                   double* __restrict__ out6) {
  pdl_wait();
  pdl_launch();
  if (threadIdx.x != 0) return;
  const Stats st = stats[blockIdx.x];
  const long long a = st.cnt[0], b = st.cnt[1], i = st.cnt[2];
  double* o = out6 + (int64_t)blockIdx.x * 6;
  o[0] = __ddiv_rn((double)(2 * i), (double)(a + b));
  o[1] = __ddiv_rn((double)i, (double)(a + b - i));
  if (a == 0 || b == 0) {
    const double v = a == 0 && b == 0 ? __longlong_as_double(0x7ff8000000000000ll) : __longlong_as_double(0x7ff0000000000000ll);
    o[2] = o[3] = o[4] = o[5] = v;
    return;
  }
  double pct[2];
  for (int dir = 0; dir < 2; ++dir) {
    long long lo, hi;
    double t = 0.0;
    percentile_ranks(st.cnt[3 + dir], q, &lo, &hi, &t);
    const double lo_v = __longlong_as_double((long long)sel[blockIdx.x * kSel + 2 * dir].prefix);
    const double hi_v = __longlong_as_double((long long)sel[blockIdx.x * kSel + 2 * dir + 1].prefix);
    pct[dir] = lo == hi ? lo_v : lerp(lo_v, hi_v, t);
  }
  o[2] = fmax(st.mx[0], st.mx[1]);
  o[3] = fmax(pct[0], pct[1]);
  o[4] = __ddiv_rn(st.sum[0], (double)st.cnt[3]);
  o[5] = __ddiv_rn(__dadd_rn(st.sum[0], st.sum[1]), (double)(st.cnt[3] + st.cnt[4]));
}

// ---- host side ----
inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

inline bool overlap(const void* a, size_t na, const void* b, size_t nb) {
  const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
  return x < y + nb && y < x + na;
}

inline bool shape_ok(int32_t items, int32_t d, int32_t h, int32_t w) {
  return items >= 1 && d >= 1 && h >= 1 && w >= 1 && (int64_t)d * h * w <= 0x7fffffff;
}

// The transform's workspace: int32 and fp64 envelope vertices, laid out like the images.
inline size_t edt_bytes(int64_t voxels) { return align256((size_t)voxels * 4) + align256((size_t)voxels * 8); }

inline int64_t chunks_of(int64_t n, int64_t chunk) { return ceil_div(n, chunk); }

struct Layout {   // mask_agreement's workspace
  size_t dist_t, dist_p, code, te, env, part, stats, sel, hist, total;
};

inline Layout layout_of(int32_t items, int32_t d, int32_t h, int32_t w) {
  const int64_t n = (int64_t)d * h * w, v = items * n;
  Layout L;
  size_t o = 0;
  L.dist_t = o; o += align256((size_t)v * 8);
  L.dist_p = o; o += align256((size_t)v * 8);
  L.code = o;   o += align256((size_t)v);
  L.te = o;     o += align256((size_t)v);
  L.env = o;    const size_t morph = mpgan_morphology_workspace(items, d, h, w);
  o += align256(edt_bytes(v) > morph ? edt_bytes(v) : morph);
  L.part = o;   o += align256((size_t)items * chunks_of(n, kChunk) * sizeof(Partial));
  L.stats = o;  o += align256((size_t)items * sizeof(Stats));
  L.sel = o;    o += align256((size_t)items * kSel * sizeof(Sel));
  L.hist = o;   o += align256((size_t)items * kSel * kBins * 4);
  L.total = o;
  return L;
}

// Shape, spacing and pointer checks shared by both entry points (MPGAN_ERR_SHAPE before any CUDA call).
static int check_common(const char* what, const void* mask, int32_t rank, int32_t items, int32_t d, int32_t h,
                        int32_t w, double sd, double sh, double sw, const void* out, const void* workspace) {
  MPGAN_REQUIRE(mask && out && workspace, MPGAN_ERR_SHAPE, "%s: null pointer", what);
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "%s: rank %d (2 or 3)", what, (int)rank);
  MPGAN_REQUIRE(items >= 1 && d >= 1 && h >= 1 && w >= 1, MPGAN_ERR_SHAPE, "%s: size items %d x (%d, %d, %d)", what,
                (int)items, (int)d, (int)h, (int)w);
  MPGAN_REQUIRE(rank == 3 || d == 1, MPGAN_ERR_SHAPE, "%s: d %d at rank 2 (must be 1)", what, (int)d);
  MPGAN_REQUIRE((int64_t)d * h * w <= 0x7fffffff, MPGAN_ERR_SHAPE, "%s: %lld voxels per image (1 .. 2^31 - 1)", what,
                (long long)d * h * w);
  const double sp[3] = {sd, sh, sw};
  for (int i = 0; i < 3; ++i)
    MPGAN_REQUIRE(sp[i] > 0.0 && isfinite(sp[i]), MPGAN_ERR_SHAPE, "%s: spacing %g (positive and finite)", what, sp[i]);
  const int64_t v = (int64_t)items * d * h * w;
  MPGAN_REQUIRE(ceil_div(v / w, kRowWarps) <= 0x7fffffff && ceil_div(v / h, kColThreads) <= 0x7fffffff &&
                    ceil_div(v / d, kColThreads) <= 0x7fffffff &&
                    items * chunks_of((int64_t)d * h * w, kChunk) <= 0x7fffffff,
                MPGAN_ERR_SHAPE, "%s: too many items", what);
  return 0;
}

// The three (rank 3) or two (rank 2) passes of the transform of `mask` (kSurface: of the complement of the surface
// mask & ~eroded) into out.
template <bool kSurface>
static int edt(const uint8_t* mask, const uint8_t* eroded, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w,
               double sd, double sh, double sw, double* out, void* env, cudaStream_t s) {
  const int64_t v = (int64_t)items * d * h * w;
  int* env_v = (int*)env;
  double* env_f = (double*)((char*)env + align256((size_t)v * 4));
  const int64_t rows = v / w;
  launch_k(edt_rows_kernel<kSurface>, (unsigned)ceil_div(rows, kRowWarps), kRowWarps * 32, 0, s, mask, eroded, rows, w,
           sw, env_v, out);
  MPGAN_CHECK_LAUNCH("edt_rows_kernel");
  const int64_t cols_y = v / h;
  launch_k(edt_cols_kernel, (unsigned)ceil_div(cols_y, kColThreads), kColThreads, 0, s, cols_y, (int)h, (int64_t)w, sh,
           rank == 2 ? 1 : 0, out, env_v, env_f);
  MPGAN_CHECK_LAUNCH("edt_cols_kernel");
  if (rank == 3) {
    const int64_t cols_z = v / d;
    launch_k(edt_cols_kernel, (unsigned)ceil_div(cols_z, kColThreads), kColThreads, 0, s, cols_z, (int)d,
             (int64_t)h * w, sd, 1, out, env_v, env_f);
    MPGAN_CHECK_LAUNCH("edt_cols_kernel");
  }
  return 0;
}

}  // namespace dist
}  // namespace mpgan

using namespace mpgan;
using namespace mpgan::dist;

extern "C" size_t mpgan_distance_transform_workspace(int32_t items, int32_t d, int32_t h, int32_t w) {
  if (!shape_ok(items, d, h, w)) return 0;
  return edt_bytes((int64_t)items * d * h * w);
}

extern "C" int mpgan_distance_transform(const uint8_t* mask, int32_t rank, int32_t items, int32_t d, int32_t h,
                                        int32_t w, double sd, double sh, double sw, double* out, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  if (int rc = check_common("distance_transform", mask, rank, items, d, h, w, sd, sh, sw, out, workspace)) return rc;
  const size_t v = (size_t)items * d * h * w, need = edt_bytes((int64_t)v);
  MPGAN_REQUIRE(workspace_bytes >= need, MPGAN_ERR_SHAPE, "distance_transform: workspace too small (%zu < %zu bytes)",
                workspace_bytes, need);
  MPGAN_REQUIRE(!overlap(mask, v, out, v * 8), MPGAN_ERR_SHAPE, "distance_transform: output overlaps the input");
  MPGAN_REQUIRE(!overlap(workspace, workspace_bytes, mask, v) && !overlap(workspace, workspace_bytes, out, v * 8),
                MPGAN_ERR_SHAPE, "distance_transform: workspace overlaps the input or the output");
  return edt<false>(mask, nullptr, rank, items, d, h, w, sd, sh, sw, out, workspace, (cudaStream_t)stream);
}

extern "C" size_t mpgan_mask_agreement_workspace(int32_t items, int32_t d, int32_t h, int32_t w) {
  if (!shape_ok(items, d, h, w)) return 0;
  return layout_of(items, d, h, w).total;
}

extern "C" int mpgan_mask_agreement(const uint8_t* pred, const uint8_t* truth, int32_t rank, int32_t items, int32_t d,
                                    int32_t h, int32_t w, double sd, double sh, double sw, int32_t connectivity,
                                    double percentile, double* out6, void* workspace, size_t workspace_bytes,
                                    void* stream) {
  MPGAN_REQUIRE(truth, MPGAN_ERR_SHAPE, "mask_agreement: null pointer");
  if (int rc = check_common("mask_agreement", pred, rank, items, d, h, w, sd, sh, sw, out6, workspace)) return rc;
  MPGAN_REQUIRE(connectivity >= 1 && connectivity <= rank, MPGAN_ERR_SHAPE,
                "mask_agreement: connectivity %d (1 .. rank %d)", (int)connectivity, (int)rank);
  MPGAN_REQUIRE(percentile >= 0.0 && percentile <= 100.0, MPGAN_ERR_SHAPE, "mask_agreement: percentile %g (0 .. 100)",
                percentile);
  const Layout L = layout_of(items, d, h, w);
  MPGAN_REQUIRE(workspace_bytes >= L.total, MPGAN_ERR_SHAPE, "mask_agreement: workspace too small (%zu < %zu bytes)",
                workspace_bytes, L.total);
  const size_t v = (size_t)items * d * h * w;
  MPGAN_REQUIRE(!overlap(out6, (size_t)items * 48, pred, v) && !overlap(out6, (size_t)items * 48, truth, v),
                MPGAN_ERR_SHAPE, "mask_agreement: output overlaps an input");
  MPGAN_REQUIRE(!overlap(workspace, workspace_bytes, pred, v) && !overlap(workspace, workspace_bytes, truth, v) &&
                    !overlap(workspace, workspace_bytes, out6, (size_t)items * 48),
                MPGAN_ERR_SHAPE, "mask_agreement: workspace overlaps an input or the output");
  cudaStream_t s = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  double* dist_t = (double*)(ws + L.dist_t);
  double* dist_p = (double*)(ws + L.dist_p);
  uint8_t* code = (uint8_t*)(ws + L.code);   // the erosion of P, then the surface codes
  uint8_t* te = (uint8_t*)(ws + L.te);
  void* env = ws + L.env;
  const size_t env_bytes = L.part - L.env;
  Partial* part = (Partial*)(ws + L.part);
  Stats* stats = (Stats*)(ws + L.stats);
  Sel* sel = (Sel*)(ws + L.sel);
  unsigned* hist = (unsigned*)(ws + L.hist);
  cudaError_t e = cudaMemsetAsync(hist, 0, (size_t)items * kSel * kBins * 4, s);
  MPGAN_REQUIRE(e == cudaSuccess, MPGAN_ERR_CUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
  // the surfaces: one erosion of each mask (the envelope region is free until the transforms run)
  if (int rc = mpgan_binary_morphology(pred, rank, items, d, h, w, connectivity, 0, 1, code, env, env_bytes, stream))
    return rc;
  if (int rc = mpgan_binary_morphology(truth, rank, items, d, h, w, connectivity, 0, 1, te, env, env_bytes, stream))
    return rc;
  if (int rc = edt<true>(truth, te, rank, items, d, h, w, sd, sh, sw, dist_t, env, s)) return rc;
  if (int rc = edt<true>(pred, code, rank, items, d, h, w, sd, sh, sw, dist_p, env, s)) return rc;
  const int64_t n = (int64_t)d * h * w;
  const int chunks = (int)chunks_of(n, kChunk);
  const double q = percentile / 100.0;
  launch_k(agree_reduce_kernel, (unsigned)(items * chunks), kThreads, 0, s, pred, truth, code, (const uint8_t*)te,
           (const double*)dist_t, (const double*)dist_p, n, chunks, part);
  MPGAN_CHECK_LAUNCH("agree_reduce_kernel");
  launch_k(agree_combine_kernel, (unsigned)items, kThreads, 0, s, (const Partial*)part, chunks, q, stats, sel);
  MPGAN_CHECK_LAUNCH("agree_combine_kernel");
  const int hchunks = (int)chunks_of(n, kHistChunk);
  for (int level = 0; level < kLevels; ++level) {
    launch_k(agree_hist_kernel, (unsigned)(items * hchunks), kThreads, 0, s, (const uint8_t*)code,
             (const double*)dist_t, (const double*)dist_p, n, hchunks, level, (const Sel*)sel, hist);
    MPGAN_CHECK_LAUNCH("agree_hist_kernel");
    launch_k(agree_select_kernel, (unsigned)items, kThreads, 0, s, level, sel, hist);
    MPGAN_CHECK_LAUNCH("agree_select_kernel");
  }
  launch_k(agree_final_kernel, (unsigned)items, 32, 0, s, (const Stats*)stats, (const Sel*)sel, q, out6);
  MPGAN_CHECK_LAUNCH("agree_final_kernel");
  return 0;
}
