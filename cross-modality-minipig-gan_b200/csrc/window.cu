// Sliding-window inference over volumes of any size (MONAI 0.4.0 `sliding_window_inference`, the call the reference's
// minipig_inference.py:110-114 leaves commented out): gather one chunk of windows from the virtually padded input, and
// blend the windows' predictions back into the unpadded output with a separable importance map.
//
// The geometry (per-dim window starts, coverage ranges and importance taps) is one caller-owned int32 table whose layout
// include/mpgan.h documents.  The host validates its host copy completely before any launch; the kernels read the device
// copy.  Rank 2 is rank 3 with a trivial leading dim (extent 1, one window, tap 1).
//
// gather: one warp per output row (window, channel, i0, i1) along the innermost dim; float4 loads and stores when the
// row lies inside the image and its source and destination are 16-byte aligned, scalar (cval outside the image) else.
// blend: gather-style, one thread per output voxel.  It reads the windows covering it (found in O(1) per dim from the
// coverage table) and sums w * y in fp64 in window order.  The denominator sum_k w factorises over the Cartesian grid
// into prod_d sum_j t_d(p_d - s_{d,j}), so no count map exists.  No atomics: the result is bit-identical run to run.
#include "common.cuh"

namespace mpgan {
namespace window {

constexpr int kHeaderWords = 16;

struct Geom {
  int s[3], roi[3], lo[3], n[3];
};

struct Layout {
  int64_t starts, cover, taps, words;   // word offsets into the table; taps are fp64 (two words each)
};

inline Layout layout_of(const Geom& g) {
  Layout l;
  l.starts = kHeaderWords;
  l.cover = l.starts + (int64_t)g.n[0] + g.n[1] + g.n[2];
  int64_t p = 0, r = 0;
  for (int d = 0; d < 3; ++d) {
    p += (int64_t)g.s[d] + (g.roi[d] - g.s[d] > 0 ? g.roi[d] - g.s[d] : 0);
    r += g.roi[d];
  }
  l.taps = l.cover + 2 * p;
  l.taps += l.taps & 1;
  l.words = l.taps + 2 * r;
  return l;
}

__global__ void __launch_bounds__(128) window_gather_kernel(const float* __restrict__ x, int channels, Geom g,
                                                            const int* __restrict__ starts, int64_t first, int rows,
                                                            float cval, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int row = blockIdx.x * blockDim.y + threadIdx.y;
  if (row >= rows) return;
  int r = row;
  const int i1 = r % g.roi[1];
  r /= g.roi[1];
  const int i0 = r % g.roi[0];
  r /= g.roi[0];
  const int c = r % channels, k = r / channels;
  const int64_t nwin = (int64_t)g.n[0] * g.n[1] * g.n[2];
  const int64_t kg = first + k;
  const int64_t b = kg / nwin;
  int w = (int)(kg - b * nwin);
  const int j2 = w % g.n[2];
  w /= g.n[2];
  const int j1 = w % g.n[1], j0 = w / g.n[1];
  const int q0 = starts[j0] + i0 - g.lo[0];
  const int q1 = starts[g.n[0] + j1] + i1 - g.lo[1];
  const int off = starts[g.n[0] + g.n[1] + j2] - g.lo[2];   // input column of the row's first element
  const int r2 = g.roi[2], s2 = g.s[2];
  float* o = out + (int64_t)row * r2;
  const bool inside = q0 >= 0 && q0 < g.s[0] && q1 >= 0 && q1 < g.s[1];
  const float* src = x + (((b * channels + c) * g.s[0] + q0) * (int64_t)g.s[1] + q1) * s2;
  if (inside && off >= 0 && off + r2 <= s2 && (r2 & 3) == 0 && (((uintptr_t)(src + off) | (uintptr_t)o) & 15) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(src + off);
    float4* o4 = reinterpret_cast<float4*>(o);
    for (int v = threadIdx.x; v < (r2 >> 2); v += 32) o4[v] = __ldg(s4 + v);
    return;
  }
  for (int i = threadIdx.x; i < r2; i += 32) {
    const int q = off + i;
    o[i] = inside && q >= 0 && q < s2 ? __ldg(src + q) : cval;
  }
}

__global__ void __launch_bounds__(128) window_blend_kernel(const float* __restrict__ pred, int channels, Geom g,
                                                           const int* __restrict__ tab, const double* __restrict__ taps,
                                                           float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int q2 = blockIdx.y * blockDim.x + threadIdx.x;
  if (q2 >= g.s[2]) return;
  int r = blockIdx.x;   // ((b * C + c) * S0 + q0) * S1 + q1
  const int q1 = r % g.s[1];
  r /= g.s[1];
  const int q0 = r % g.s[0];
  r /= g.s[0];
  const int c = r % channels, b = r / channels;

  const int* st0 = tab + kHeaderWords;
  const int* st1 = st0 + g.n[0];
  const int* st2 = st1 + g.n[1];
  const int* cv0 = st2 + g.n[2];                 // coverage pairs per padded coordinate; padded extent = max(s, roi)
  const int* cv1 = cv0 + 2 * max(g.s[0], g.roi[0]);
  const int* cv2 = cv1 + 2 * max(g.s[1], g.roi[1]);
  const double* t0 = taps;
  const double* t1 = t0 + g.roi[0];
  const double* t2 = t1 + g.roi[1];

  const int p0 = q0 + g.lo[0], p1 = q1 + g.lo[1], p2 = q2 + g.lo[2];
  const int f0 = cv0[2 * p0], l0 = cv0[2 * p0 + 1];
  const int f1 = cv1[2 * p1], l1 = cv1[2 * p1 + 1];
  const int f2 = cv2[2 * p2], l2 = cv2[2 * p2 + 1];
  const int64_t vol = (int64_t)g.roi[0] * g.roi[1] * g.roi[2];
  const int64_t nwin = (int64_t)g.n[0] * g.n[1] * g.n[2];
  const int64_t win_stride = channels * vol;   // elements between consecutive windows

  double d0 = 0.0, d1 = 0.0, d2 = 0.0, num = 0.0;
  for (int j = f1; j <= l1; ++j) d1 += t1[p1 - st1[j]];
  for (int j = f2; j <= l2; ++j) d2 += t2[p2 - st2[j]];
  for (int j0 = f0; j0 <= l0; ++j0) {
    const int i0 = p0 - st0[j0];
    const double w0 = t0[i0];
    d0 += w0;
    for (int j1 = f1; j1 <= l1; ++j1) {
      const int i1 = p1 - st1[j1];
      const double w01 = w0 * t1[i1];
      const int64_t k = (int64_t)b * nwin + ((int64_t)j0 * g.n[1] + j1) * g.n[2];
      const float* base = pred + k * win_stride + c * vol + ((int64_t)i0 * g.roi[1] + i1) * g.roi[2];
      for (int j2 = f2; j2 <= l2; ++j2) {
        const int i2 = p2 - st2[j2];
        num = fma(w01 * t2[i2], (double)__ldg(base + j2 * win_stride + i2), num);
      }
    }
  }
  out[(int64_t)blockIdx.x * g.s[2] + q2] = (float)(num / (d0 * d1 * d2));
}

// Validate the host copy of the table against (rank, size, roi) semantics; on success fill *g.
int check_geom(const char* what, const int32_t* t, int64_t words, const void* dev, Geom* g, Layout* lay) {
  MPGAN_REQUIRE(t && dev, MPGAN_ERR_SHAPE, "%s: null geometry table", what);
  MPGAN_REQUIRE(((uintptr_t)dev & 7) == 0, MPGAN_ERR_SHAPE, "%s: device geometry table not 8-byte aligned", what);
  MPGAN_REQUIRE(words >= kHeaderWords, MPGAN_ERR_SHAPE, "%s: geometry table of %lld words (header alone is %d)", what,
                (long long)words, kHeaderWords);
  const int rank = t[0];
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "%s: rank %d (2 or 3)", what, rank);
  for (int d = 0; d < 3; ++d) {
    g->s[d] = t[1 + d];
    g->roi[d] = t[4 + d];
    g->lo[d] = t[7 + d];
    g->n[d] = t[10 + d];
    MPGAN_REQUIRE(g->s[d] > 0 && g->roi[d] > 0 && g->n[d] > 0, MPGAN_ERR_SHAPE,
                  "%s: dim %d: size %d, roi %d, windows %d must be positive", what, d, g->s[d], g->roi[d], g->n[d]);
    const int diff = g->roi[d] > g->s[d] ? g->roi[d] - g->s[d] : 0;
    MPGAN_REQUIRE(g->lo[d] == diff / 2, MPGAN_ERR_SHAPE, "%s: dim %d: lo %d, expected %d for size %d and roi %d", what, d,
                  g->lo[d], diff / 2, g->s[d], g->roi[d]);
    MPGAN_REQUIRE(g->s[d] <= (1 << 22) && g->roi[d] <= (1 << 22), MPGAN_ERR_SHAPE, "%s: dim %d: extent above 2^22",
                  what, d);
  }
  MPGAN_REQUIRE(rank == 3 || (g->s[0] == 1 && g->roi[0] == 1 && g->n[0] == 1), MPGAN_ERR_SHAPE,
                "%s: rank 2 needs a trivial leading dim (size 1, roi 1, one window)", what);
  *lay = layout_of(*g);
  MPGAN_REQUIRE(words == lay->words, MPGAN_ERR_SHAPE, "%s: geometry table of %lld words, its header implies %lld", what,
                (long long)words, (long long)lay->words);
  const int32_t* st = t + lay->starts;
  const int32_t* cv = t + lay->cover;
  const double* tp = reinterpret_cast<const double*>(t + lay->taps);
  for (int d = 0; d < 3; ++d) {
    const int pd = g->s[d] + (g->roi[d] > g->s[d] ? g->roi[d] - g->s[d] : 0);
    for (int j = 0; j < g->n[d]; ++j) {
      MPGAN_REQUIRE(st[j] >= 0 && st[j] + g->roi[d] <= pd, MPGAN_ERR_SHAPE,
                    "%s: dim %d: window %d starts at %d, past padded extent %d - roi %d", what, d, j, st[j], pd, g->roi[d]);
      MPGAN_REQUIRE(j == 0 || st[j] > st[j - 1], MPGAN_ERR_SHAPE, "%s: dim %d: window starts not increasing", what, d);
    }
    for (int p = 0; p < pd; ++p) {
      const int f = cv[2 * p], l = cv[2 * p + 1];
      const bool in_image = p >= g->lo[d] && p < g->lo[d] + g->s[d];
      if (!in_image) continue;   // the blend never reads coverage of padding
      // starts increase, so [f, l] are exactly the windows covering p iff these four hold
      MPGAN_REQUIRE(f >= 0 && f <= l && l < g->n[d] && st[l] <= p && p < st[f] + g->roi[d] &&
                        (f == 0 || st[f - 1] + g->roi[d] <= p) && (l == g->n[d] - 1 || st[l + 1] > p),
                    MPGAN_ERR_SHAPE, "%s: dim %d: coverage [%d, %d] of padded coordinate %d is not the windows covering it",
                    what, d, f, l, p);
    }
    for (int i = 0; i < g->roi[d]; ++i)
      MPGAN_REQUIRE(tp[i] > 0.0 && tp[i] <= 1.0, MPGAN_ERR_SHAPE, "%s: dim %d: tap %d = %g not in (0, 1]", what, d, i,
                    tp[i]);
    st += g->n[d];
    cv += 2 * pd;
    tp += g->roi[d];
  }
  return 0;
}

}  // namespace window
}  // namespace mpgan

using namespace mpgan;

extern "C" int mpgan_window_gather(const float* x, int32_t batch, int32_t channels, const int32_t* geom,
                                   const int32_t* geom_dev, int64_t geom_words, int64_t first, int64_t count, float cval,
                                   float* out, void* stream) {
  using namespace mpgan::window;
  Geom g;
  Layout lay;
  MPGAN_REQUIRE(x && out, MPGAN_ERR_SHAPE, "window_gather: null pointer");
  if (int rc = check_geom("window_gather", geom, geom_words, geom_dev, &g, &lay)) return rc;
  MPGAN_REQUIRE(batch > 0 && channels > 0, MPGAN_ERR_SHAPE, "window_gather: batch %d, channels %d", (int)batch,
                (int)channels);
  const int64_t total = (int64_t)batch * g.n[0] * g.n[1] * g.n[2];
  MPGAN_REQUIRE(first >= 0 && count > 0 && first <= total && count <= total - first, MPGAN_ERR_SHAPE,
                "window_gather: windows [%lld, %lld) outside the %lld windows of %d images", (long long)first,
                (long long)(first + count), (long long)total, (int)batch);
  const int64_t rows = count * channels * g.roi[0] * g.roi[1];
  MPGAN_REQUIRE(rows <= 0x7fffffff, MPGAN_ERR_SHAPE, "window_gather: too many rows");
  launch_k(window_gather_kernel, dim3((unsigned)ceil_div(rows, 4)), dim3(32, 4), 0, (cudaStream_t)stream, x,
           (int)channels, g, (const int*)(geom_dev + lay.starts), first, (int)rows, cval, out);
  MPGAN_CHECK_LAUNCH("window_gather_kernel");
  return 0;
}

extern "C" int mpgan_window_blend(const float* pred, int32_t batch, int32_t channels, const int32_t* geom,
                                  const int32_t* geom_dev, int64_t geom_words, float* out, void* stream) {
  using namespace mpgan::window;
  Geom g;
  Layout lay;
  MPGAN_REQUIRE(pred && out, MPGAN_ERR_SHAPE, "window_blend: null pointer");
  if (int rc = check_geom("window_blend", geom, geom_words, geom_dev, &g, &lay)) return rc;
  MPGAN_REQUIRE(batch > 0 && channels > 0, MPGAN_ERR_SHAPE, "window_blend: batch %d, channels %d", (int)batch,
                (int)channels);
  const int64_t rows = (int64_t)batch * channels * g.s[0] * g.s[1];
  MPGAN_REQUIRE(rows <= 0x7fffffff, MPGAN_ERR_SHAPE, "window_blend: too many rows");
  launch_k(window_blend_kernel, dim3((unsigned)rows, (unsigned)ceil_div(g.s[2], 128)), dim3(128), 0,
           (cudaStream_t)stream, pred, (int)channels, g, (const int*)geom_dev,
           reinterpret_cast<const double*>(geom_dev + lay.taps), out);
  MPGAN_CHECK_LAUNCH("window_blend_kernel");
  return 0;
}
