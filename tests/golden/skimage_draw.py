"""TEST INFRASTRUCTURE ONLY -- never imported by the product (pylinac_b200/).

``skimage.draw.disk`` and ``skimage.draw.ellipse`` restated from scikit-image's source (skimage/draw/draw.py: ``ellipse`` and its
``_ellipse_in_shape``; ``disk(center, radius, shape)`` is ``ellipse(r, c, radius, radius, shape)``), for the disk goldens that run the
unmodified reference ``DiskROI`` (core/roi.py:134-150).  scikit-image is not installed here, so parity with the real library is
UNPINNED at this boundary, like the other restated skimage functions in oracle/skimage_shim.py; everything downstream of the pixel
set (statistics, wrap-around, errors, contrast, MTF) is pinned by tests/golden/disk_roi_golden.npz.  Only rotation 0 is exercised.
"""
from __future__ import annotations

import types

import numpy as np


def _ellipse_in_shape(shape, center, radii, rotation=0.0):
    """Row / column indices (np.nonzero order) of the pixels of an ``shape`` box inside the ellipse: distances < 1."""
    r_lim, c_lim = np.ogrid[0:float(shape[0]), 0:float(shape[1])]
    r_org, c_org = center
    r_rad, c_rad = radii
    rotation %= np.pi
    sin_alpha, cos_alpha = np.sin(rotation), np.cos(rotation)
    r, c = (r_lim - r_org), (c_lim - c_org)
    distances = ((r * cos_alpha + c * sin_alpha) / r_rad) ** 2 + ((r * sin_alpha - c * cos_alpha) / c_rad) ** 2
    return np.nonzero(distances < 1)


def ellipse(r, c, r_radius, c_radius, shape=None, rotation=0.0):
    """skimage.draw.ellipse: bounding box ceil(center - rotated radii) .. floor(center + rotated radii), clipped to ``shape`` only when
    it is given (without it the indices may be negative or beyond the image)."""
    center = np.array([r, c])
    radii = np.array([r_radius, c_radius])
    rotation %= np.pi
    r_radius_rot = abs(r_radius * np.cos(rotation)) + c_radius * np.sin(rotation)
    c_radius_rot = r_radius * np.sin(rotation) + abs(c_radius * np.cos(rotation))
    radii_rot = np.array([r_radius_rot, c_radius_rot])
    upper_left = np.ceil(center - radii_rot).astype(int)
    lower_right = np.floor(center + radii_rot).astype(int)
    if shape is not None:
        upper_left = np.maximum(upper_left, np.array([0, 0]))
        lower_right = np.minimum(lower_right, np.array(shape[:2]) - 1)
    shifted_center = center - upper_left
    bounding_shape = lower_right - upper_left + 1
    rr, cc = _ellipse_in_shape(bounding_shape, shifted_center, radii, rotation)
    rr.flags.writeable = True
    cc.flags.writeable = True
    rr += upper_left[0]
    cc += upper_left[1]
    return rr, cc


def disk(center, radius, *, shape=None):
    """skimage.draw.disk(center=(row, col), radius, shape=None)"""
    r, c = center
    return ellipse(r, c, radius, radius, shape)


def install():
    """Serve ``skimage.draw`` to the reference's core/roi.py (after oracle.refstub.import_reference())."""
    import pylinac.core.roi as rroi

    rroi.draw = types.SimpleNamespace(disk=disk, ellipse=ellipse)
