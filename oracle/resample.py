"""TEST INFRASTRUCTURE (oracle): numpy fp64 restatement of linear resampling between physical grids.  Only tests/ and
tools/ may import this module.

Follows ITK 5.1's ``ResampleImageFilter`` + ``IdentityTransform`` + ``LinearInterpolateImageFunction`` on float pixels
as ITK documents them (the reference's ``ResampleT1T2d``, code/GAN/transforms.py:79-213).  ITK is not available here,
so this is a restatement of the semantics pinned in include/mpgan.h, not a copy of ITK; bit-parity with ITK is not
claimed (ITK forms the continuous index incrementally along a row and inverts its matrix with vnl).  Per output voxel
with ITK index i = (i_x, i_y, i_z), every operation a separate fp64 rounding (elementwise numpy ufuncs, no ``@``,
``einsum`` or ``dot``, which may reorder or fuse):
  p_k = ((o_out_k + M_out[k,0] i_x) + M_out[k,1] i_y) + M_out[k,2] i_z            TransformIndexToPhysicalPoint
  c_k = ((N_in[k,0] (p_0 - o_in_0)) + N_in[k,1] (p_1 - o_in_1)) + N_in[k,2] (p_2 - o_in_2)   ...ToContinuousIndex
  inside iff -0.5 <= c_k < n_k - 0.5 on every axis, else default_value;
  per axis b = max(floor(c), 0), d = c - b (d <= 0 -> 0), upper neighbour min(b + 1, n - 1), unused at d = 0;
  lerps a + (b - a) d along x, then y, then z; one rounding to float32.
M_out = D_out diag(S_out) and N_in = inverse(D_in diag(S_in)) come from ``mpgan.transforms.ImageGeometry``, the one
place they are computed, so the kernel and this module see the same bits.  Rank 2 is rank 3 with a trivial z.
"""
import numpy as np


def _lift(geometry, matrix):
    """(size[3], origin[3], matrix 3x3) in ITK axis order, a rank-2 geometry with the identity's z row and column."""
    r = geometry.rank
    m = np.eye(3)
    m[:r, :r] = matrix
    return (tuple(geometry.size) + (1,) * (3 - r), tuple(geometry.origin) + (0.0,) * (3 - r), m)


def continuous_index(source, target):
    """(3, Z, Y, X) fp64: the continuous source index (ITK axis order k = x, y, z) of every target voxel."""
    size_o, o_out, m = _lift(target, target.index_to_physical())
    _, o_in, n = _lift(source, source.physical_to_index())
    iz, iy, ix = np.meshgrid(*(np.arange(s, dtype=np.float64) for s in size_o[::-1]), indexing="ij")
    p = [((o_out[k] + m[k, 0] * ix) + m[k, 1] * iy) + m[k, 2] * iz for k in range(3)]
    q = [p[k] - o_in[k] for k in range(3)]
    return np.stack([((n[k, 0] * q[0]) + n[k, 1] * q[1]) + n[k, 2] * q[2] for k in range(3)])


def inside(c, size):
    """Half-open inside test of continuous indices c (3, ...) against a size[3] in ITK axis order."""
    with np.errstate(invalid="ignore"):
        return np.all([(c[k] >= -0.5) & (c[k] < size[k] - 0.5) for k in range(3)], axis=0)


def interpolate(x3, c, size):
    """fp64 linear interpolation of x3 (items, nz, ny, nx) at continuous indices c (3, ...), clamped as the semantics
    state; values at outside indices are meaningless.  Returns (items, ...)."""
    x3 = np.asarray(x3, dtype=np.float64)
    lo, hi, w = [], [], []
    for k in range(3):
        ck = np.nan_to_num(c[k], nan=0.0)
        b = np.clip(np.maximum(np.floor(ck), 0.0), 0, size[k] - 1)
        d = ck - b
        lo.append(b.astype(np.int64))
        hi.append(np.minimum(lo[k] + 1, size[k] - 1))
        w.append(np.where(d > 0, d, 0.0))

    def at(zi, yi, xi):
        return x3[:, zi, yi, xi]

    def lerp(a, b, d):
        return np.where(d > 0, a + (b - a) * d, a)

    with np.errstate(invalid="ignore", over="ignore"):
        def plane(zi):
            r0 = lerp(at(zi, lo[1], lo[0]), at(zi, lo[1], hi[0]), w[0])
            r1 = lerp(at(zi, hi[1], lo[0]), at(zi, hi[1], hi[0]), w[0])
            return lerp(r0, r1, w[1])
        return lerp(plane(lo[2]), plane(hi[2]), w[2])


def resample(image, source, target, default_value=0.0):
    """image (*lead, *source.shape) -> (*lead, *target.shape) float32."""
    image = np.asarray(image, dtype=np.float32)
    lead = image.shape[:image.ndim - source.rank]
    size_in = _lift(source, source.index_to_physical())[0]
    x3 = image.reshape((-1,) + size_in[::-1])
    c = continuous_index(source, target)
    val = interpolate(x3, c, size_in)
    out = np.where(inside(c, size_in), val, np.float64(np.float32(default_value))).astype(np.float32)
    return out.reshape(lead + tuple(target.shape))
