"""Relative and moments-based MTF -- mirror of ``pylinac.core.mtf`` (core/mtf.py:32-305): ``MTF`` / ``PeakValleyMTF``, ``moments_mtf``,
``moments_fwhm`` and ``MomentMTF``.

These are scalar host computations on ROI results: the maxima / minima (``MTF``) and means / standard deviations (``MomentMTF``) of
high-contrast disks or rectangles, which the device computes (``epid_disk_roi_stats`` / ``epid_roi_stats``).  ``relative_resolution``
restates scipy's ``interp1d(..., fill_value="extrapolate")`` in numpy with scipy's own arithmetic, so the package keeps scipy out of
its import graph.  ``EdgeSpreadFunctionMTF`` and the plotting methods are not mirrored."""
from __future__ import annotations

import math
import warnings
from collections.abc import Sequence

import numpy as np

from .contrast import michelson


def _interp1d_extrapolate(x, y, x_new) -> np.ndarray:
    """scipy.interpolate.interp1d(x, y, fill_value="extrapolate")(x_new), kind "linear": the points sorted by x (stable), the segment
    found by searchsorted and clipped to the first / last segment outside the data, then de Boor's form
    (x_new - x_lo) / (x_hi - x_lo) * y_hi + (x_hi - x_new) / (x_hi - x_lo) * y_lo as scipy evaluates it."""
    x = np.array(x)
    y = np.array(y)
    ind = np.argsort(x, kind="mergesort")
    x, y = x[ind], y[ind]
    if not issubclass(y.dtype.type, np.inexact):
        y = y.astype(np.float64)
    xn = np.asarray(x_new)
    if not issubclass(xn.dtype.type, np.inexact):
        xn = xn.astype(np.float64)
    shape = xn.shape
    xn = xn.ravel()
    idx = np.searchsorted(x, xn).clip(1, len(x) - 1).astype(int)
    x_lo, x_hi, y_lo, y_hi = x[idx - 1], x[idx], y[idx - 1], y[idx]
    y_new = (xn - x_lo) / (x_hi - x_lo) * y_hi + (x_hi - xn) / (x_hi - x_lo) * y_lo
    return y_new.reshape(shape)


class MTF:
    """Relative MTF from the maxima and minima of line-pair regions (core/mtf.py:32-112)."""

    def __init__(self, lp_spacings: Sequence[float], lp_maximums: Sequence[float], lp_minimums: Sequence[float]):
        self.spacings = lp_spacings
        self.maximums = lp_maximums
        self.minimums = lp_minimums
        if len(lp_spacings) != len(lp_maximums) != len(lp_minimums):
            raise ValueError("The number of MTF spacings, maximums, and minimums must be equal.")
        if len(lp_spacings) < 2 or len(lp_maximums) < 2 or len(lp_minimums) < 2:
            raise ValueError("The number of MTF spacings, maximums, and minimums must be greater than 1.")
        self.mtfs = {}
        self.norm_mtfs = {}
        for spacing, max, min in zip(lp_spacings, lp_maximums, lp_minimums):
            arr = np.array((max, min))
            self.mtfs[spacing] = michelson(arr)
        self.mtfs = {k: v for k, v in sorted(self.mtfs.items(), key=lambda x: x[0])}
        for key, value in self.mtfs.items():
            self.norm_mtfs[key] = value / self.mtfs[lp_spacings[0]]       # normalised to the FIRST given spacing, as the reference
        max_delta = np.max(np.diff(list(self.norm_mtfs.values())))
        if max_delta > 0:
            warnings.warn("The MTF does not drop monotonically; be sure the ROIs are correctly aligned.")

    def relative_resolution(self, x: float = 50) -> float:
        """The line-pair value at x % of the relative MTF; 0 <= x <= 100 (core/mtf.py:82-101)."""
        if not 0 <= x <= 100:
            raise ValueError(f"x must be between 0 and 100; got {x}")
        mtf = _interp1d_extrapolate(list(self.norm_mtfs.values()), list(self.norm_mtfs.keys()), x / 100)
        if mtf > max(self.spacings):
            warnings.warn(f"MTF resolution wasn't calculated for {x}% that was asked for. The value returned is an extrapolation. "
                          "Use a higher % MTF to get a non-interpolated value.")
        return float(mtf)

    @classmethod
    def from_high_contrast_diskset(cls, spacings: Sequence[float], diskset) -> MTF:
        """From HighContrastDiskROI / RectangleROI objects: their max and min (core/mtf.py:103-112)."""
        maximums = [roi.max for roi in diskset]
        minimums = [roi.min for roi in diskset]
        return cls(spacings, maximums, minimums)


class PeakValleyMTF(MTF):
    pass


def moments_mtf(mean: float, std: float) -> float:
    """Hander et al 1997, eq. 8 (core/mtf.py:194-201)."""
    return math.sqrt(2 * (std**2 - mean)) / mean


def moments_fwhm(width: float, mean: float, std: float) -> float:
    """Hander et al 1997, eq. A8 (core/mtf.py:204-220)."""
    return 1.058 * width * math.sqrt(np.log(mean / (math.sqrt(2 * (std**2 - mean)))))


class MomentMTF:
    """Moments-based MTF and FWHM per line-pair frequency (core/mtf.py:223-260)."""

    mtfs: dict[float, float]
    fwhms: dict[float, float]

    def __init__(self, lpmms: Sequence[float], means: Sequence[float], stds: Sequence[float]):
        self.mtfs = {}
        self.fwhms = {}
        for lpmm, mean, std in zip(lpmms, means, stds):
            bar_width = 1 / (2 * lpmm)  # lp is 2 bars
            self.mtfs[lpmm] = moments_mtf(mean, std)
            self.fwhms[lpmm] = moments_fwhm(bar_width, mean, std)

    @classmethod
    def from_high_contrast_diskset(cls, lpmms: Sequence[float], diskset) -> MomentMTF:
        """From HighContrastDiskROI objects: their mean and std (core/mtf.py:253-260)."""
        means = [roi.mean for roi in diskset]
        stds = [roi.std for roi in diskset]
        return cls(lpmms, means, stds)
