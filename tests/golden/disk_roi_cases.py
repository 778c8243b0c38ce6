"""Seeded frames and disk layouts for the DiskROI / contrast / MTF goldens (tests/golden/disk_roi_golden.npz).

The frames are built here with numpy alone so that the GPU tests can rebuild them without the reference: a uint16 phantom-like image
(rows != columns, so an error on the wrong axis shows), and float64 / float32 frames made from it by ``ground()`` and ``normalize()``
as planar_imaging prepares its images (array - array.min(), then / array.max(); make_disk_roi_golden.py checks that the reference's
ArrayImage.ground / normalize give the same arrays)."""
from __future__ import annotations

import numpy as np

SHAPE = (360, 400)
KINDS = ("u16", "f64", "f32")
PERCENTILES = (0, 2.5, 50, 97.5, 100)
DPI = 30.48          # 1.2 px / mm

# name -> (x, y, radius): fractional radii, centres on .5 (boundary ties), integer centre + radius (an empty last row / column of the
# bounding box), disks over the top / left edges (numpy wraps the negative indices), over the bottom / right edges (IndexError), an
# empty disk, and one too large to stage in shared memory
DISKS = {
    "qc3": (120.3, 95.7, 19.0),
    "half_centre": (200.5, 180.5, 7.5),
    "int_tie": (50.0, 60.0, 5.0),
    "odd_even_a": (300.25, 80.75, 3.6),
    "odd_even_b": (301.0, 81.5, 4.5),
    "tiny": (33.3, 44.4, 1.2),
    "wrap_top": (150.2, 3.4, 9.0),
    "wrap_left": (2.0, 200.0, 6.5),
    "wrap_corner": (1.5, 2.5, 5.0),
    "oob_bottom": (150.0, 357.0, 6.0),
    "oob_right": (398.0, 100.0, 4.0),
    "empty": (10.5, 10.5, 0.5),
    "r60": (260.3, 170.8, 60.0),
    "large": (200.0, 180.0, 150.0),
}
ERROR_DISKS = ("oob_bottom", "oob_right")
SMALL_DISKS = tuple(k for k in DISKS if k not in ("r60", "large"))     # pixel values stored for these

# LowContrastDiskROI: (disk, contrast_reference or None); every contrast method is applied to each
LOW_CONTRAST = (("qc3", 0.62), ("half_centre", 0.35), ("tiny", None), ("r60", 0.5))
CONTRAST_METHODS = ("Michelson", "Weber", "Ratio", "Root Mean Square", "Difference")

# MTF / MomentMTF from high-contrast disk sets on the uint16 frame: (spacings, disk centres, radius)
MTF_SETS = {
    "monotonic": ((0.1, 0.2, 0.3, 0.4), ((60, 250), (110, 250), (160, 250), (210, 250)), 10.0),
    "non_monotonic": ((0.1, 0.2, 0.3, 0.4), ((60, 250), (160, 250), (110, 250), (210, 250)), 10.0),
}
MTF_RESOLUTIONS = (90, 50, 30, 10, 0)

# DiskROIMetric / RectangleROIMetric through image.compute: pixel and physical (mm) versions; compute runs twice so the in-place
# dpmm scaling of from_physical shows
METRICS = {
    "disk_px": ("DiskROIMetric", False, dict(radius=12.5, center=(140.0, 120.0))),
    "disk_mm": ("DiskROIMetric", True, dict(radius_mm=8.0, center_mm=(100.0, 80.0))),
    "rect_px": ("RectangleROIMetric", False, dict(width=30.0, height=20.0, center=(220.0, 140.0))),
    "rect_mm": ("RectangleROIMetric", True, dict(width_mm=20.0, height_mm=12.0, center_mm=(150.0, 110.0))),
}


def raw_frame() -> np.ndarray:
    """uint16 [360, 400]: a smooth field, a few disks of different contrast and a bar pattern, Gaussian noise."""
    rng = np.random.default_rng(2024)
    h, w = SHAPE
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float64)
    img = 18000 + 6000 * np.exp(-(((yy - 180) / 160) ** 2 + ((xx - 200) / 180) ** 2))
    for (x, y, r, a) in ((120.3, 95.7, 19, 2500), (200.5, 180.5, 9, -1800), (260.3, 170.8, 45, 900), (33.3, 44.4, 3, 4000)):
        img += a * (((xx - x) ** 2 + (yy - y) ** 2) < r * r)
    for k, (x, y) in enumerate(((60, 250), (110, 250), (160, 250), (210, 250))):      # bar groups of decreasing modulation
        bars = np.sin(2 * np.pi * (xx - x) / (6 - k)) > 0
        img += (9000 - 2000 * k) * (bars & (np.abs(xx - x) < 12) & (np.abs(yy - y) < 12))
    img += rng.normal(0, 120, SHAPE)
    return img.clip(0, 65535).astype(np.uint16)


def frame(kind: str) -> np.ndarray:
    raw = raw_frame()
    if kind == "u16":
        return raw
    a = raw.astype(np.float32) if kind == "f32" else raw
    a = a - a.min() + 0           # core/array_utils.py ground()
    return a / a.max()            # core/array_utils.py normalize(): float64 for the uint16 frame, float32 for the float32 one
