// Connected components and binary morphology of foreground masks: scipy.ndimage's label, binary_fill_holes,
// binary_erosion and binary_dilation under generate_binary_structure(rank, connectivity), and the largest component.
// include/mpgan.h pins the semantics.
//
// Labelling is a block-based union-find with a fixed number of launches (no convergence loop, so it can be captured
// in a CUDA graph):
//   1. cc_local_kernel: one CTA per tile of 1024 voxels unites every "in" voxel with its backward neighbours (those of
//      smaller linear index) inside the tile, in shared memory, and writes each voxel's tile root as a linear index.
//   2. cc_merge_kernel: voxels on a tile's backward faces unite with their neighbours in other tiles, in global memory.
//   3. cc_flatten_kernel: every voxel's parent becomes its root (and, per entry point, root counts, component sizes or
//      face marks are gathered in the same pass).
// A union always hangs the larger root under the smaller one (atomicMin), so whatever order the atomics land in, the
// root of a component is its smallest linear index: the result is deterministic and numbers components as scipy does.
// label then flags the roots, scans the flags per image over linear chunks (cc_scan_kernel) and gives every voxel its
// root's rank + 1.  Background voxels have parent -1 and label 0.
#include "common.cuh"

namespace mpgan {
namespace morph {

constexpr int kTile = 1024;                    // voxels per union-find tile, one thread each; the width is 32
constexpr int kTW = 32;
constexpr int kThreads = 256;                  // chunk kernels: kPer voxels per thread, coalesced
constexpr int kPer = 8;
constexpr int kChunk = kThreads * kPer;
constexpr int kScanThreads = 1024;

struct Img {
  int rank, conn, d, h, w, n;
};

__device__ __forceinline__ int ld_volatile(const int* p) { return *(const volatile int*)p; }

// Root of x with path halving.  Safe while other threads unite: a parent only ever moves to one of its ancestors, and
// the CAS only replaces x -> p by x -> parent(p) when x still points at p, so no link is lost.
__device__ __forceinline__ int find_root(int* p, int x) {
  int px = ld_volatile(p + x);
  while (px != x) {
    const int gp = ld_volatile(p + px);
    if (gp != px) atomicCAS(p + x, px, gp);
    x = gp;
    px = ld_volatile(p + x);
  }
  return x;
}

// Union of the sets of a and b: the larger root is hung under the smaller one.  When atomicMin finds that the larger
// root has meanwhile got a parent, the union continues with that parent (Playne and Hawick 2018).
__device__ __forceinline__ void unite(int* p, int a, int b) {
  while (true) {
    a = find_root(p, a);
    b = find_root(p, b);
    if (a == b) return;
    if (a > b) {
      const int t = a;
      a = b;
      b = t;
    }
    const int old = atomicMin(p + b, a);
    if (old == b) return;
    b = old;
  }
}

// Backward neighbours in the structure: offsets whose first non-zero component is negative, with |dz|+|dy|+|dx| <= conn
// (3, 9 or 13 of them at rank 3; 2 or 4 at rank 2).  f(dz, dy, dx) for each.
template <class F>
__device__ __forceinline__ void for_backward(const Img& im, F&& f) {
#pragma unroll
  for (int dz = -1; dz <= 0; ++dz) {
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
#pragma unroll
      for (int dx = -1; dx <= 1; ++dx) {
        const bool back = dz < 0 || (dz == 0 && (dy < 0 || (dy == 0 && dx < 0)));
        if (back && (dz == 0 || im.rank == 3) && -dz + abs(dy) + abs(dx) <= im.conn) f(dz, dy, dx);
      }
    }
  }
}

// The tile of this CTA: (item, origin) and this thread's tile-local coordinates.  Rank 3 tiles are 4 x 8 x 32, rank 2
// tiles 1 x 32 x 32.
struct TilePos {
  int item, z0, y0, x0, tz, ty, tx, td, th;
};
__device__ __forceinline__ TilePos tile_pos(const Img& im, int tiles_z, int tiles_y, int tiles_x) {
  TilePos t;
  t.td = im.rank == 3 ? 4 : 1;
  t.th = kTile / kTW / t.td;
  const int per_item = tiles_z * tiles_y * tiles_x;
  t.item = blockIdx.x / per_item;
  int r = blockIdx.x % per_item;
  t.x0 = (r % tiles_x) * kTW;
  r /= tiles_x;
  t.y0 = (r % tiles_y) * t.th;
  t.z0 = (r / tiles_y) * t.td;
  t.tx = threadIdx.x % kTW;
  t.ty = (threadIdx.x / kTW) % t.th;
  t.tz = threadIdx.x / (kTW * t.th);
  return t;
}

// Step 1.  "in" is mask != 0, or mask == 0 with kInvert (the background, for fill_holes).  parent[g] = the linear index
// of g's tile root (the tile's smallest voxel of g's tile-local component), -1 outside.  zero_at_roots (nullable) is
// zeroed at tile roots: the global roots are among them, so a later per-root counter starts at 0 without a memset.
template <bool kInvert>
__global__ void __launch_bounds__(kTile) cc_local_kernel(const uint8_t* __restrict__ mask, Img im, int tiles_z,
                                                         int tiles_y, int tiles_x, int* __restrict__ parent,
                                                         int* __restrict__ zero_at_roots) {
  __shared__ int sp[kTile];
  pdl_wait();
  pdl_launch();
  const TilePos t = tile_pos(im, tiles_z, tiles_y, tiles_x);
  const int z = t.z0 + t.tz, y = t.y0 + t.ty, x = t.x0 + t.tx;
  const bool valid = z < im.d && y < im.h && x < im.w;
  const int64_t base = (int64_t)t.item * im.n;
  const int g = valid ? (z * im.h + y) * im.w + x : 0;
  const bool in = valid && ((__ldg(mask + base + g) != 0) != kInvert);
  const int me = threadIdx.x;
  sp[me] = in ? me : -1;
  __syncthreads();
  if (in) {
    for_backward(im, [&](int dz, int dy, int dx) {
      const int nz = t.tz + dz, ny = t.ty + dy, nx = t.tx + dx;
      if (nz >= 0 && ny >= 0 && ny < t.th && nx >= 0 && nx < kTW) {   // outside the image: sp is -1 there
        const int nb = (nz * t.th + ny) * kTW + nx;
        if (sp[nb] >= 0) unite(sp, me, nb);
      }
    });
  }
  __syncthreads();
  if (!valid) return;
  int root = -1;
  if (in) {
    const int r = find_root(sp, me);
    root = ((t.z0 + r / (kTW * t.th)) * im.h + (t.y0 + (r / kTW) % t.th)) * im.w + (t.x0 + r % kTW);
    if (zero_at_roots && r == me) zero_at_roots[base + g] = 0;
  }
  parent[base + g] = root;
}

// Step 2: unions across tile faces, in global memory.  Only voxels with a backward neighbour outside their tile work.
template <bool kInvert>
__global__ void __launch_bounds__(kTile) cc_merge_kernel(const uint8_t* __restrict__ mask, Img im, int tiles_z,
                                                         int tiles_y, int tiles_x, int* __restrict__ parent) {
  pdl_wait();
  pdl_launch();
  const TilePos t = tile_pos(im, tiles_z, tiles_y, tiles_x);
  const bool face = (im.rank == 3 && (t.tz == 0 || t.ty == t.th - 1)) || t.ty == 0 || t.tx == 0 || t.tx == kTW - 1;
  const int z = t.z0 + t.tz, y = t.y0 + t.ty, x = t.x0 + t.tx;
  if (!face || z >= im.d || y >= im.h || x >= im.w) return;
  const int64_t base = (int64_t)t.item * im.n;
  const int g = (z * im.h + y) * im.w + x;
  if ((__ldg(mask + base + g) != 0) == kInvert) return;
  int* p = parent + base;
  for_backward(im, [&](int dz, int dy, int dx) {
    const int nz = t.tz + dz, ny = t.ty + dy, nx = t.tx + dx;
    const bool other_tile = nz < 0 || ny < 0 || ny >= t.th || nx < 0 || nx >= kTW;
    if (other_tile && z + dz >= 0 && y + dy >= 0 && y + dy < im.h && x + dx >= 0 && x + dx < im.w) {
      const int nb = ((z + dz) * im.h + (y + dy)) * im.w + (x + dx);
      if ((__ldg(mask + base + nb) != 0) != kInvert) unite(p, g, nb);
    }
  });
}

enum { kCountRoots = 0, kSizes = 1, kMarkFaces = 2 };

// Step 3 over linear chunks of kChunk voxels: parent[g] = root(g), and
//   kCountRoots: chunk_roots[item][chunk] = the roots in the chunk (for the scan of label);
//   kSizes:      aux[root] += 1 per voxel (warp-aggregated integer atomics): component sizes;
//   kMarkFaces:  aux[root] = 1 for every voxel on a face of the image: components that touch a face.
template <int kMode>
__global__ void __launch_bounds__(kThreads) cc_flatten_kernel(Img im, int chunks, int* __restrict__ parent,
                                                              int* __restrict__ aux, int* __restrict__ chunk_roots) {
  pdl_wait();
  pdl_launch();
  const int item = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  int* p = parent + (int64_t)item * im.n;
  int* a = kMode == kCountRoots ? nullptr : aux + (int64_t)item * im.n;
  const int g0 = chunk * kChunk, lim = min(kChunk, im.n - g0);
  int roots = 0;
#pragma unroll 1
  for (int k = 0; k < kPer; ++k) {
    const int off = k * kThreads + threadIdx.x, g = g0 + off;
    int r = off < lim ? p[g] : -1;
    if (r >= 0) {
      if (r == g) {
        ++roots;
      } else {
        int q = p[r];
        while (q != r) {
          r = q;
          q = p[r];
        }
        p[g] = r;
      }
    }
    if constexpr (kMode == kSizes) {
      const unsigned same = __match_any_sync(0xffffffffu, r);
      if (r >= 0 && (threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(a + r, __popc(same));
    } else if constexpr (kMode == kMarkFaces) {
      if (r >= 0) {
        const int x = g % im.w, y = (g / im.w) % im.h, z = g / im.w / im.h;
        if (x == 0 || x == im.w - 1 || y == 0 || y == im.h - 1 || (im.rank == 3 && (z == 0 || z == im.d - 1))) a[r] = 1;
      }
    }
  }
  if constexpr (kMode == kCountRoots) {
    __shared__ int s[kThreads / 32];
    const int v = __reduce_add_sync(0xffffffffu, roots);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int i = 0; i < kThreads / 32; ++i) tot += s[i];
      chunk_roots[blockIdx.x] = tot;
    }
  }
}

// One CTA per item: chunk_roots[item][*] -> its exclusive prefix sums in place, count[item] = the total.
__global__ void __launch_bounds__(kScanThreads) cc_scan_kernel(int chunks, int* __restrict__ chunk_roots,
                                                               int32_t* __restrict__ count) {
  __shared__ int s[kScanThreads / 32];
  pdl_wait();
  pdl_launch();
  int* c = chunk_roots + (int64_t)blockIdx.x * chunks;
  const int per = (chunks + kScanThreads - 1) / kScanThreads;
  const int c0 = min(chunks, (int)threadIdx.x * per), c1 = min(chunks, c0 + per);
  int sum = 0;
  for (int i = c0; i < c1; ++i) sum += c[i];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s[warp] = incl;
  __syncthreads();
  int before = 0, total = 0;
  for (int i = 0; i < kScanThreads / 32; ++i) {
    before += i < warp ? s[i] : 0;
    total += s[i];
  }
  int run = before + incl - sum;
  for (int i = c0; i < c1; ++i) {
    const int v = c[i];
    c[i] = run;
    run += v;
  }
  if (threadIdx.x == 0) count[blockIdx.x] = total;
}

// labels[root] = its rank among the item's roots in raster order + 1 (chunk offset from the scan, then the roots before
// it in the chunk, counted per pass with warp ballots).
__global__ void __launch_bounds__(kThreads) cc_root_labels_kernel(Img im, int chunks, const int* __restrict__ parent,
                                                                  const int* __restrict__ chunk_offsets,
                                                                  int32_t* __restrict__ labels) {
  __shared__ int s[kThreads / 32];
  pdl_wait();
  pdl_launch();
  const int item = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const int* p = parent + (int64_t)item * im.n;
  int32_t* l = labels + (int64_t)item * im.n;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g0 = chunk * kChunk, lim = min(kChunk, im.n - g0);
  int run = chunk_offsets[blockIdx.x];
#pragma unroll 1
  for (int k = 0; k < kPer; ++k) {
    const int off = k * kThreads + threadIdx.x, g = g0 + off;
    const bool root = off < lim && p[g] == g;
    const unsigned b = __ballot_sync(0xffffffffu, root);
    if (lane == 0) s[warp] = __popc(b);
    __syncthreads();
    int before = 0, total = 0;
#pragma unroll
    for (int i = 0; i < kThreads / 32; ++i) {
      before += i < warp ? s[i] : 0;
      total += s[i];
    }
    if (root) l[g] = run + before + __popc(b & ((1u << lane) - 1)) + 1;
    run += total;
    __syncthreads();
  }
}

// labels[g] = labels[root(g)], 0 in the background.
__global__ void __launch_bounds__(kThreads) cc_propagate_kernel(Img im, int chunks, const int* __restrict__ parent,
                                                                int32_t* __restrict__ labels) {
  pdl_wait();
  pdl_launch();
  const int item = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const int* p = parent + (int64_t)item * im.n;
  int32_t* l = labels + (int64_t)item * im.n;
  const int g0 = chunk * kChunk, lim = min(kChunk, im.n - g0);
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    const int off = k * kThreads + threadIdx.x, g = g0 + off;
    if (off >= lim) break;
    const int r = p[g];
    if (r != g) l[g] = r < 0 ? 0 : l[r];
  }
}

// best[item] = max over roots of (size << 32) | (0xffffffff - root): the largest component, ties to the smallest root.
__global__ void __launch_bounds__(kThreads) cc_best_kernel(Img im, int chunks, const int* __restrict__ parent,
                                                           const int* __restrict__ sizes,
                                                           unsigned long long* __restrict__ best) {
  pdl_wait();
  pdl_launch();
  const int item = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const int64_t base = (int64_t)item * im.n;
  const int g0 = chunk * kChunk, lim = min(kChunk, im.n - g0);
  unsigned long long m = 0;
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    const int off = k * kThreads + threadIdx.x, g = g0 + off;
    if (off < lim && parent[base + g] == g) {
      const unsigned long long v = ((unsigned long long)(unsigned)sizes[base + g] << 32) | (0xffffffffu - (unsigned)g);
      m = v > m ? v : m;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long v = __shfl_xor_sync(0xffffffffu, m, o);
    m = v > m ? v : m;
  }
  if ((threadIdx.x & 31) == 0 && m) atomicMax(best + item, m);
}

// out = in the item's largest component (empty when the item has none).
__global__ void __launch_bounds__(kThreads) cc_keep_best_kernel(Img im, int chunks, const int* __restrict__ parent,
                                                                const unsigned long long* __restrict__ best,
                                                                uint8_t* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int item = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const int64_t base = (int64_t)item * im.n;
  const unsigned long long b = best[item];
  const int keep = b ? (int)(0xffffffffu - (unsigned)(b & 0xffffffffu)) : -1;
  const int g0 = chunk * kChunk, lim = min(kChunk, im.n - g0);
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    const int off = k * kThreads + threadIdx.x, g = g0 + off;
    if (off >= lim) break;
    const int r = parent[base + g];
    out[base + g] = r >= 0 && r == keep;
  }
}

// out = mask | (background component touching no face): bg_parent holds the flattened roots of the background's
// components (-1 on the mask), marks[root] != 0 where the component touches a face.
__global__ void __launch_bounds__(kThreads) cc_fill_kernel(Img im, int chunks, const int* __restrict__ bg_parent,
                                                           const int* __restrict__ marks, uint8_t* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int item = blockIdx.x / chunks, chunk = blockIdx.x % chunks;
  const int64_t base = (int64_t)item * im.n;
  const int g0 = chunk * kChunk, lim = min(kChunk, im.n - g0);
#pragma unroll
  for (int k = 0; k < kPer; ++k) {
    const int off = k * kThreads + threadIdx.x, g = g0 + off;
    if (off >= lim) break;
    const int r = bg_parent[base + g];
    out[base + g] = r < 0 || marks[base + r] == 0;
  }
}

// ---- erosion / dilation: one 3^rank stencil pass restricted to the structure, border value 0 ----
// Each thread writes kV consecutive voxels of a row: kV = 16 with 16-byte loads and stores when every row is 16-byte
// aligned, else 1.  A neighbour row is read as bits, bit j = voxel x0 - 1 + j, with its left and right neighbours.
__device__ __forceinline__ unsigned nz_bits4(unsigned v) {   // bit i = (byte i != 0)
  const unsigned m = __vcmpne4(v, 0u) & 0x01010101u;
  return (m * 0x01020408u) >> 24;
}
__device__ __forceinline__ unsigned bytes_of4(unsigned b) {   // byte i = bit i
  return (b & 1u) | ((b & 2u) << 7) | ((b & 4u) << 14) | ((b & 8u) << 21);
}

template <int kV>
__global__ void __launch_bounds__(kThreads) morph_kernel(const uint8_t* __restrict__ in, Img im, int erode,
                                                         int blocks_per_item, uint8_t* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int item = blockIdx.x / blocks_per_item;
  const int groups_per_row = im.w / kV;
  const int64_t q64 = (int64_t)(blockIdx.x % blocks_per_item) * kThreads + threadIdx.x;
  if (q64 >= (int64_t)im.d * im.h * groups_per_row) return;
  const int q = (int)q64;
  const int x0 = (q % groups_per_row) * kV, row = q / groups_per_row, y = row % im.h, z = row / im.h;
  const int64_t base = (int64_t)item * im.n;
  const unsigned all = kV == 16 ? 0xffffu : 1u;
  unsigned acc = erode ? all : 0u;
#pragma unroll
  for (int dz = -1; dz <= 1; ++dz) {
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
      const int m = abs(dz) + abs(dy);
      if ((dz != 0 && im.rank == 2) || m > im.conn) continue;
      unsigned r = 0;   // bits 0 .. kV + 1
      const int zz = z + dz, yy = y + dy;
      if (zz >= 0 && zz < im.d && yy >= 0 && yy < im.h) {
        const uint8_t* src = in + base + ((int64_t)zz * im.h + yy) * im.w;
        if constexpr (kV == 16) {
          const uint4 v = __ldg(reinterpret_cast<const uint4*>(src + x0));
          r = (nz_bits4(v.x) | (nz_bits4(v.y) << 4) | (nz_bits4(v.z) << 8) | (nz_bits4(v.w) << 12)) << 1;
        } else {
          r = (unsigned)(__ldg(src + x0) != 0) << 1;
        }
        if (x0 > 0) r |= (unsigned)(__ldg(src + x0 - 1) != 0);
        if (x0 + kV < im.w) r |= (unsigned)(__ldg(src + x0 + kV) != 0) << (kV + 1);
      }
      unsigned c = (r >> 1) & all;
      if (m + 1 <= im.conn) c = erode ? c & r & (r >> 2) : c | r | (r >> 2);
      acc = erode ? acc & c : acc | (c & all);
    }
  }
  uint8_t* dst = out + base + ((int64_t)z * im.h + y) * im.w + x0;
  if constexpr (kV == 16) {
    *reinterpret_cast<uint4*>(dst) = make_uint4(bytes_of4(acc), bytes_of4(acc >> 4), bytes_of4(acc >> 8),
                                                bytes_of4(acc >> 12));
  } else {
    *dst = (uint8_t)(acc & 1u);
  }
}

// ---- host side ----
struct Plan {
  Img im;
  int items, tiles_z, tiles_y, tiles_x, chunks;
  int* parent;                    // workspace: items x n int32
  int* aux;                       // workspace: items x n int32 (sizes, face marks, or the erosion ping-pong buffer)
  int* chunk_roots;               // workspace: items x chunks int32
  unsigned long long* best;       // workspace: items uint64
};

inline size_t align16(size_t b) { return (b + 15) & ~(size_t)15; }

inline size_t workspace_bytes(int64_t items, int64_t n) {
  const int64_t chunks = (n + kChunk - 1) / kChunk;
  return 2 * align16((size_t)(items * n) * 4) + align16((size_t)(items * chunks) * 4) + (size_t)items * 8;
}

inline bool overlap(const void* a, size_t na, const void* b, size_t nb) {
  const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
  return x < y + nb && y < x + na;
}

// Validates every argument (MPGAN_ERR_SHAPE before any CUDA call) and lays out the workspace.
static int plan_of(const char* what, const uint8_t* mask, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w,
                   int32_t connectivity, const void* out, size_t out_elem, void* workspace, size_t ws_bytes, Plan* pl) {
  MPGAN_REQUIRE(mask && out && workspace, MPGAN_ERR_SHAPE, "%s: null pointer", what);
  MPGAN_REQUIRE(rank == 2 || rank == 3, MPGAN_ERR_SHAPE, "%s: rank %d (2 or 3)", what, (int)rank);
  MPGAN_REQUIRE(connectivity >= 1 && connectivity <= rank, MPGAN_ERR_SHAPE, "%s: connectivity %d (1 .. rank %d)", what,
                (int)connectivity, (int)rank);
  MPGAN_REQUIRE(items >= 1 && d >= 1 && h >= 1 && w >= 1, MPGAN_ERR_SHAPE, "%s: size items %d x (%d, %d, %d)", what,
                (int)items, (int)d, (int)h, (int)w);
  MPGAN_REQUIRE(rank == 3 || d == 1, MPGAN_ERR_SHAPE, "%s: d %d at rank 2 (must be 1)", what, (int)d);
  const int64_t n = (int64_t)d * h * w;
  MPGAN_REQUIRE(n <= 0x7fffffff, MPGAN_ERR_SHAPE, "%s: %lld voxels per image (1 .. 2^31 - 1)", what, (long long)n);
  MPGAN_REQUIRE(ws_bytes >= workspace_bytes(items, n), MPGAN_ERR_SHAPE, "%s: workspace too small (%zu < %zu bytes)", what,
                ws_bytes, workspace_bytes(items, n));
  const size_t in_bytes = (size_t)items * n;
  MPGAN_REQUIRE(!overlap(mask, in_bytes, out, in_bytes * out_elem), MPGAN_ERR_SHAPE, "%s: output overlaps the input", what);
  MPGAN_REQUIRE(!overlap(workspace, ws_bytes, mask, in_bytes) && !overlap(workspace, ws_bytes, out, in_bytes * out_elem),
                MPGAN_ERR_SHAPE, "%s: workspace overlaps the input or the output", what);
  Plan& p = *pl;
  p.im = Img{rank, connectivity, d, h, w, (int)n};
  p.items = items;
  const int td = rank == 3 ? 4 : 1, th = kTile / kTW / td;
  p.tiles_z = (int)ceil_div(d, td);
  p.tiles_y = (int)ceil_div(h, th);
  p.tiles_x = (int)ceil_div(w, kTW);
  p.chunks = (int)ceil_div(n, kChunk);
  const int64_t tiles = (int64_t)p.tiles_z * p.tiles_y * p.tiles_x;
  MPGAN_REQUIRE(items * tiles <= 0x7fffffff && items * (int64_t)p.chunks <= 0x7fffffff, MPGAN_ERR_SHAPE,
                "%s: too many items", what);
  char* ws = (char*)workspace;
  p.parent = (int*)ws;
  ws += align16(in_bytes * 4);
  p.aux = (int*)ws;
  ws += align16(in_bytes * 4);
  p.chunk_roots = (int*)ws;
  ws += align16((size_t)items * p.chunks * 4);
  p.best = (unsigned long long*)ws;
  return 0;
}

// Steps 1-3 for the "in" voxels (kInvert: the background); kMode selects what the flatten pass gathers.
template <bool kInvert, int kMode>
static int components(const uint8_t* mask, const Plan& p, cudaStream_t s) {
  const unsigned tile_grid = (unsigned)((int64_t)p.items * p.tiles_z * p.tiles_y * p.tiles_x);
  launch_k(cc_local_kernel<kInvert>, tile_grid, kTile, 0, s, mask, p.im, p.tiles_z, p.tiles_y, p.tiles_x, p.parent,
           kMode == kCountRoots ? (int*)nullptr : p.aux);
  MPGAN_CHECK_LAUNCH("cc_local_kernel");
  launch_k(cc_merge_kernel<kInvert>, tile_grid, kTile, 0, s, mask, p.im, p.tiles_z, p.tiles_y, p.tiles_x, p.parent);
  MPGAN_CHECK_LAUNCH("cc_merge_kernel");
  launch_k(cc_flatten_kernel<kMode>, (unsigned)((int64_t)p.items * p.chunks), kThreads, 0, s, p.im, p.chunks, p.parent,
           p.aux, p.chunk_roots);
  MPGAN_CHECK_LAUNCH("cc_flatten_kernel");
  return 0;
}

}  // namespace morph
}  // namespace mpgan

using namespace mpgan;
using namespace mpgan::morph;

extern "C" size_t mpgan_morphology_workspace(int32_t items, int32_t d, int32_t h, int32_t w) {
  if (items < 1 || d < 1 || h < 1 || w < 1 || (int64_t)d * h * w > 0x7fffffff) return 0;
  return workspace_bytes(items, (int64_t)d * h * w);
}

extern "C" int mpgan_label(const uint8_t* mask, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w,
                           int32_t connectivity, int32_t* labels, int32_t* count, void* workspace, size_t workspace_bytes,
                           void* stream) {
  MPGAN_REQUIRE(count, MPGAN_ERR_SHAPE, "label: null pointer");
  Plan p;
  if (int rc = plan_of("label", mask, rank, items, d, h, w, connectivity, labels, 4, workspace, workspace_bytes, &p))
    return rc;
  MPGAN_REQUIRE(!overlap(count, (size_t)items * 4, mask, (size_t)items * p.im.n) &&
                    !overlap(count, (size_t)items * 4, labels, (size_t)items * p.im.n * 4) &&
                    !overlap(count, (size_t)items * 4, workspace, workspace_bytes),
                MPGAN_ERR_SHAPE, "label: count overlaps another buffer");
  cudaStream_t s = (cudaStream_t)stream;
  if (int rc = components<false, kCountRoots>(mask, p, s)) return rc;
  launch_k(cc_scan_kernel, (unsigned)items, kScanThreads, 0, s, p.chunks, p.chunk_roots, count);
  MPGAN_CHECK_LAUNCH("cc_scan_kernel");
  const unsigned grid = (unsigned)((int64_t)items * p.chunks);
  launch_k(cc_root_labels_kernel, grid, kThreads, 0, s, p.im, p.chunks, (const int*)p.parent,
           (const int*)p.chunk_roots, labels);
  MPGAN_CHECK_LAUNCH("cc_root_labels_kernel");
  launch_k(cc_propagate_kernel, grid, kThreads, 0, s, p.im, p.chunks, (const int*)p.parent, labels);
  MPGAN_CHECK_LAUNCH("cc_propagate_kernel");
  return 0;
}

extern "C" int mpgan_largest_component(const uint8_t* mask, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w,
                                       int32_t connectivity, uint8_t* out, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  Plan p;
  if (int rc = plan_of("largest_component", mask, rank, items, d, h, w, connectivity, out, 1, workspace, workspace_bytes,
                       &p))
    return rc;
  cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = cudaMemsetAsync(p.best, 0, (size_t)items * sizeof(unsigned long long), s);
  MPGAN_REQUIRE(e == cudaSuccess, MPGAN_ERR_CUDA, "cudaMemsetAsync: %s", cudaGetErrorString(e));
  if (int rc = components<false, kSizes>(mask, p, s)) return rc;
  const unsigned grid = (unsigned)((int64_t)items * p.chunks);
  launch_k(cc_best_kernel, grid, kThreads, 0, s, p.im, p.chunks, (const int*)p.parent, (const int*)p.aux, p.best);
  MPGAN_CHECK_LAUNCH("cc_best_kernel");
  launch_k(cc_keep_best_kernel, grid, kThreads, 0, s, p.im, p.chunks, (const int*)p.parent,
           (const unsigned long long*)p.best, out);
  MPGAN_CHECK_LAUNCH("cc_keep_best_kernel");
  return 0;
}

extern "C" int mpgan_fill_holes(const uint8_t* mask, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w,
                                int32_t connectivity, uint8_t* out, void* workspace, size_t workspace_bytes,
                                void* stream) {
  Plan p;
  if (int rc = plan_of("fill_holes", mask, rank, items, d, h, w, connectivity, out, 1, workspace, workspace_bytes, &p))
    return rc;
  cudaStream_t s = (cudaStream_t)stream;
  if (int rc = components<true, kMarkFaces>(mask, p, s)) return rc;
  launch_k(cc_fill_kernel, (unsigned)((int64_t)items * p.chunks), kThreads, 0, s, p.im, p.chunks, (const int*)p.parent,
           (const int*)p.aux, out);
  MPGAN_CHECK_LAUNCH("cc_fill_kernel");
  return 0;
}

extern "C" int mpgan_binary_morphology(const uint8_t* mask, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w,
                                       int32_t connectivity, int32_t op, int32_t iterations, uint8_t* out,
                                       void* workspace, size_t workspace_bytes, void* stream) {
  MPGAN_REQUIRE(op == 0 || op == 1, MPGAN_ERR_SHAPE, "binary_morphology: op %d (0 erode, 1 dilate)", (int)op);
  MPGAN_REQUIRE(iterations >= 1, MPGAN_ERR_SHAPE, "binary_morphology: iterations %d (>= 1)", (int)iterations);
  Plan p;
  if (int rc = plan_of("binary_morphology", mask, rank, items, d, h, w, connectivity, out, 1, workspace, workspace_bytes,
                       &p))
    return rc;
  cudaStream_t s = (cudaStream_t)stream;
  uint8_t* tmp = (uint8_t*)p.aux;   // 16-byte aligned
  const bool vec = w % 16 == 0 && ((uintptr_t)mask & 15) == 0 && ((uintptr_t)out & 15) == 0;
  const int64_t groups = (int64_t)d * h * (vec ? w / 16 : w);
  const int bpi = (int)ceil_div(groups, kThreads);
  MPGAN_REQUIRE((int64_t)items * bpi <= 0x7fffffff, MPGAN_ERR_SHAPE, "binary_morphology: too many items");
  const uint8_t* src = mask;
  for (int it = 1; it <= iterations; ++it) {   // the last pass writes `out`
    uint8_t* dst = (iterations - it) % 2 == 0 ? out : tmp;
    if (vec) {
      launch_k(morph_kernel<16>, (unsigned)(items * bpi), kThreads, 0, s, src, p.im, op == 0 ? 1 : 0, bpi, dst);
    } else {
      launch_k(morph_kernel<1>, (unsigned)(items * bpi), kThreads, 0, s, src, p.im, op == 0 ? 1 : 0, bpi, dst);
    }
    MPGAN_CHECK_LAUNCH("morph_kernel");
    src = dst;
  }
  return 0;
}
