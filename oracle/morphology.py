"""TEST INFRASTRUCTURE (oracle): connected components and binary morphology of masks, a thin layer over scipy.ndimage.
Only tests/ and tools/ may import this module.

include/mpgan.h pins the semantics; restated here:
  * images: the last ``spatial_dims`` (2 or 3, default min(ndim, 3)) dims are spatial, every leading index is an
    independent image; non-zero is "in".  At rank 3 an image of depth 1 has every voxel on a face.
  * structure: ``generate_binary_structure(rank, connectivity)``, connectivity 1..rank (1 by default, as in scipy).
  * label: scipy's labels (components numbered 1..k in raster order of their first voxel) and the count per image.
  * largest_component: the component with the most voxels; ties go to the lowest label (np.argmax of
    np.bincount(labels)[1:]); an empty image stays empty.
  * fill_holes: ``binary_fill_holes(mask, structure)``.
  * binary_erosion / binary_dilation: scipy's with the structure, ``iterations >= 1`` and ``border_value=0``.
  * foreground_mask: Otsu's mask (oracle/masked_metrics.py), then the largest component, then hole filling.
"""
import numpy as np
from scipy import ndimage

from . import masked_metrics as omm


def structure(rank, connectivity=1):
    return ndimage.generate_binary_structure(rank, connectivity)


def _images(mask, spatial_dims):
    """(bool images stacked on one leading axis, leading shape, rank)."""
    m = np.asarray(mask).astype(bool)
    nd = spatial_dims or min(m.ndim, 3)
    return m.reshape((-1,) + m.shape[m.ndim - nd:]), m.shape[:m.ndim - nd], nd


def label(mask, connectivity=1, spatial_dims=None):
    """(int32 labels of the mask's shape, int32 counts of the leading shape)."""
    ims, lead, nd = _images(mask, spatial_dims)
    labels = np.zeros(ims.shape, np.int32)
    counts = np.zeros(len(ims), np.int32)
    for i, im in enumerate(ims):
        labels[i], counts[i] = ndimage.label(im, structure(nd, connectivity))
    return labels.reshape(np.shape(mask)), counts.reshape(lead)


def _largest(lab):
    if lab.max() == 0:
        return np.zeros(lab.shape, bool)
    return lab == int(np.argmax(np.bincount(lab.ravel())[1:])) + 1


def largest_component(mask, connectivity=1, spatial_dims=None):
    return _per_image(lambda im, nd: _largest(ndimage.label(im, structure(nd, connectivity))[0]), mask, spatial_dims)


def _per_image(fn, mask, spatial_dims):
    ims, _, nd = _images(mask, spatial_dims)
    out = np.zeros(ims.shape, bool)
    for i, im in enumerate(ims):
        out[i] = fn(im, nd)
    return out.reshape(np.shape(mask))


def fill_holes(mask, connectivity=1, spatial_dims=None):
    return _per_image(lambda im, nd: ndimage.binary_fill_holes(im, structure(nd, connectivity)), mask, spatial_dims)


def fill_holes_by_components(mask, connectivity=1, spatial_dims=None):
    """The equivalence the kernel implements: the mask plus every background component, under the same structure,
    that touches no face of the image."""
    def fill(im, nd):
        lab, _ = ndimage.label(~im, structure(nd, connectivity))
        face = np.zeros(im.shape, bool)
        for ax in range(nd):
            idx = [slice(None)] * nd
            for end in (0, -1):
                idx[ax] = end
                face[tuple(idx)] = True
        touching = np.unique(lab[face])
        return im | ((lab > 0) & ~np.isin(lab, touching))
    return _per_image(fill, mask, spatial_dims)


def binary_erosion(mask, iterations=1, connectivity=1, spatial_dims=None):
    return _per_image(lambda im, nd: ndimage.binary_erosion(im, structure(nd, connectivity), iterations=iterations,
                                                            border_value=0), mask, spatial_dims)


def binary_dilation(mask, iterations=1, connectivity=1, spatial_dims=None):
    return _per_image(lambda im, nd: ndimage.binary_dilation(im, structure(nd, connectivity), iterations=iterations,
                                                             border_value=0), mask, spatial_dims)


def foreground_mask(x, largest=False, fill=False, connectivity=1):
    """threshold (Otsu), then the largest component, then hole filling, per image of the last min(ndim, 3) dims."""
    m = omm.foreground_mask(x)
    if largest:
        m = largest_component(m, connectivity)
    if fill:
        m = fill_holes(m, connectivity)
    return m
