"""Regions of interest -- mirror of ``pylinac.core.roi``: ``bbox_center``, the disk family ``DiskROI`` / ``LowContrastDiskROI`` /
``HighContrastDiskROI`` (core/roi.py:21-479) and ``RectangleROI`` (core/roi.py:481-706).  Plotting is out of scope.

RectangleROI: the pixel selection is skimage.draw.polygon's in the reference (``pixels_flat``); here the statistics are device
reductions over the same pixel set (``epid_roi_stats``, csrc/roi.cu: integer pixel coordinates inside or on the boundary of the corner
polygon the reference builds, clipped to the image).  ``pixel_array`` (non-rotated ROIs) is a numpy view like the reference's.

Disks: the reference samples ``array[skimage.draw.disk((y, x), r)]`` -- unclipped, so rows / columns in [-dim, -1] wrap to the far
edge and anything beyond is an IndexError -- and reduces it with numpy.  Here the device selects the same pixels and returns the
moments and exact order statistics of every disk in one launch (``epid_disk_roi_stats``) or the gathered pixels themselves
(``epid_disk_roi_pixels``); the host never rasterises a disk.  ``sample_disks_batch`` evaluates many disks on many frames at once."""
from __future__ import annotations

import numpy as np

from .. import _native as nat
from .contrast import Contrast, contrast, michelson, ratio, rms, visibility, weber
from .geometry import Circle, Point, Rectangle


def bbox_center(region) -> Point:
    """The centre of a region's bounding box (``region.bbox`` = (min_row, min_col, max_row, max_col)), core/roi.py:21-36."""
    bbox = region.bbox
    y = abs(bbox[0] - bbox[2]) / 2 + min(bbox[0], bbox[2])
    x = abs(bbox[1] - bbox[3]) / 2 + min(bbox[1], bbox[3])
    return Point(x, y)


def _device_frames(a) -> np.ndarray:
    a = np.asarray(getattr(a, "array", a))
    return a if a.dtype in nat._NP2DT else a.astype(np.float64)


def sample_disks_batch(frames, centers, radii, percentiles=()) -> dict:
    """Every disk on every frame in one launch: frames [n, H, W] (or [H, W], or a device-resident ``_native.Batch``), centers a sequence
    of Points or (x, y) pairs, radii one per disk (or one for all).  -> dict of [n, k] float64 arrays: count, mean, std, min, max, median
    (what ``DiskROI`` reports for each disk) and "percentile" [n, k, p] (``LowContrastDiskROI.percentile`` for each p).  A disk without
    pixels has count 0 and NaN statistics; a disk over the bottom or right edge raises IndexError, as the reference's indexing does."""
    pts = [Point(c) for c in centers]
    xy = np.array([[p.x, p.y] for p in pts], dtype=np.float64).reshape(-1, 2)
    f = frames if isinstance(frames, nat.Batch) else _device_frames(frames)
    return nat.disk_roi_stats(nat.Context.default(), f, xy, radii, percentiles)


class DiskROI(Circle):
    """A disk-shaped region of interest (core/roi.py:39-188).  One device launch computes and caches every statistic of the disk."""

    @classmethod
    def from_phantom_center(cls, array: np.ndarray, angle: float, roi_radius: float, dist_from_center: float, phantom_center):
        center = cls._get_shifted_center(angle, dist_from_center, phantom_center)
        return cls(array=array, center=center, radius=roi_radius)

    def __init__(self, array: np.ndarray, radius: float, center: Point):
        super().__init__(center_point=center, radius=radius)
        self._array = array
        self._stats = None
        self._pixels = None

    @staticmethod
    def _get_shifted_center(angle: float, dist_from_center: float, phantom_center: Point) -> Point:
        """The center of the ROI; corrects for phantom dislocation and roll."""
        y_shift = np.sin(np.deg2rad(angle)) * dist_from_center
        x_shift = np.cos(np.deg2rad(angle)) * dist_from_center
        return Point(phantom_center.x + x_shift, phantom_center.y + y_shift)

    def _frame(self) -> np.ndarray:
        return _device_frames(self._array)

    def _empty(self) -> np.ndarray:
        """What ``circle_mask()`` is for a disk without pixels: the numpy reductions below run on it to give the reference's NaN,
        warning or exception."""
        return np.asarray(getattr(self._array, "array", self._array))[:0, :0].ravel()

    def _compute(self) -> dict:
        if self._stats is None:
            out = nat.disk_roi_stats(nat.Context.default(), self._frame(), [[self.center.x, self.center.y]], [self.radius])
            self._stats = {k: float(v[0, 0]) for k, v in out.items() if k != "percentile"}
        return self._stats

    def _stat(self, name: str, empty) -> float:
        s = self._compute()
        return s[name] if s["count"] > 0 else float(empty(self._empty()))

    @property
    def pixel_values(self) -> np.ndarray:
        """The disk's pixel values in the reference's order (``circle_mask()``)."""
        if self._pixels is None:
            a = np.asarray(getattr(self._array, "array", self._array))
            v = nat.disk_roi_pixels(nat.Context.default(), self._frame(), 0, (self.center.x, self.center.y), self.radius)
            self._pixels = v.astype(a.dtype, copy=False)
        return self._pixels

    @property
    def pixel_value(self) -> float:
        """The median pixel value of the ROI."""
        return self._stat("median", np.median)

    @property
    def mean(self) -> float:
        """The mean value within the ROI."""
        return self._stat("mean", np.mean)

    @property
    def std(self) -> float:
        """The (population) standard deviation of the pixel values."""
        return self._stat("std", np.std)

    @property
    def min(self) -> float:
        """The min value within the ROI (ValueError for a disk without pixels, as numpy's)."""
        return self._stat("min", np.min)

    @property
    def max(self) -> float:
        """The max value within the ROI (ValueError for a disk without pixels, as numpy's)."""
        return self._stat("max", np.max)

    def circle_mask(self) -> np.ndarray:
        """The pixel values inside the disk (core/roi.py:134-138)."""
        return self.pixel_values

    def masked_array(self) -> np.ndarray:
        """An array of the image's shape with the disk's pixels (clipped to the image) and NaN elsewhere (core/roi.py:140-150).  The
        fill is the reference's np.full(shape, np.nan, dtype), so an integer image gets whatever numpy's NaN cast gives (0)."""
        a = np.asarray(getattr(self._array, "array", self._array))
        img = np.full(a.shape, np.nan, dtype=a.dtype)
        vals, rr, cc = nat.disk_roi_pixels(nat.Context.default(), self._frame(), 0, (self.center.x, self.center.y), self.radius, clip=True,
                                           indices=True)
        img[rr, cc] = vals
        return img

    def percentile(self, percentile: float) -> float:
        """The pixel value at the given percentile (np.percentile, linear; core/roi.py:406-408)."""
        if self._compute()["count"] == 0:
            return float(np.percentile(self._empty(), percentile))
        out = nat.disk_roi_stats(nat.Context.default(), self._frame(), [[self.center.x, self.center.y]], [self.radius], [percentile])
        return float(out["percentile"][0, 0, 0])

    def as_dict(self) -> dict:
        """Convert to dict. Useful for dataclasses/Result"""
        data = super().as_dict()
        data.update({"median": self.pixel_value, "std": self.std})
        return data


class LowContrastDiskROI(DiskROI):
    """A low-contrast disk: contrast against a reference value, visibility and pass / fail (core/roi.py:191-408)."""

    contrast_threshold: float | None
    cnr_threshold: float | None
    contrast_reference: float | None

    @classmethod
    def from_phantom_center(cls, array, angle: float, roi_radius: float, dist_from_center: float, phantom_center,
                            contrast_threshold: float | None = None, contrast_reference: float | None = None,
                            cnr_threshold: float | None = None, contrast_method: str = Contrast.MICHELSON,
                            visibility_threshold: float | None = 0.1):
        center = cls._get_shifted_center(angle, dist_from_center, phantom_center)
        return cls(array=array, radius=roi_radius, center=center, contrast_threshold=contrast_threshold,
                   contrast_reference=contrast_reference, cnr_threshold=cnr_threshold, contrast_method=contrast_method,
                   visibility_threshold=visibility_threshold)

    def __init__(self, array, radius: float, center: Point, contrast_threshold: float | None = None,
                 contrast_reference: float | None = None, cnr_threshold: float | None = None, contrast_method: str = Contrast.MICHELSON,
                 visibility_threshold: float = 0.1):
        super().__init__(array, radius, center=center)
        self.contrast_threshold = contrast_threshold
        self.cnr_threshold = cnr_threshold
        self.contrast_reference = contrast_reference
        self.contrast_method = contrast_method
        self.visibility_threshold = visibility_threshold

    @property
    def _contrast_array(self) -> np.ndarray:
        return np.array((self.pixel_value, self.contrast_reference))

    @property
    def signal_to_noise(self) -> float:
        """The signal-to-noise ratio. Cast to numpy first to use numpy overflow handling."""
        return float(np.array(self.pixel_value) / self.std)

    @property
    def contrast_to_noise(self) -> float:
        """The contrast to noise ratio of the ROI. Cast to numpy first to use numpy overflow handling."""
        return float(np.array(self.contrast) / self.std)

    @property
    def michelson(self) -> float:
        return michelson(self._contrast_array)

    @property
    def weber(self) -> float:
        return weber(feature=self.pixel_value, background=self.contrast_reference)

    @property
    def rms(self) -> float:
        return rms(self._contrast_array)

    @property
    def ratio(self) -> float:
        # the reference passes the 2-element array as the only argument (core/roi.py:320-323): a TypeError there and here
        return ratio(self._contrast_array)

    @property
    def contrast(self) -> float:
        """The contrast of the disk by the constructor's contrast method."""
        return contrast(self._contrast_array, self.contrast_method)

    @property
    def cnr_constant(self) -> float:
        """The contrast-to-noise value times the disk diameter."""
        return self.contrast_to_noise * self.diameter

    @property
    def visibility(self) -> float:
        """Rose-model visibility of the disk (core/contrast.py:18-40)."""
        return visibility(array=self._contrast_array, radius=self.radius, std=self.std, algorithm=self.contrast_method)

    @property
    def contrast_constant(self) -> float:
        """The contrast value times the disk diameter."""
        return self.contrast * self.diameter

    @property
    def passed(self) -> bool:
        return self.contrast > self.contrast_threshold

    @property
    def passed_visibility(self) -> bool:
        return self.visibility > self.visibility_threshold

    @property
    def passed_contrast_constant(self) -> bool:
        return self.contrast_constant > self.contrast_threshold

    @property
    def passed_cnr_constant(self) -> bool:
        return self.cnr_constant > self.cnr_threshold

    @property
    def plot_color(self) -> str:
        return "green" if self.passed_visibility else "red"

    @property
    def plot_color_constant(self) -> str:
        return "green" if self.passed_contrast_constant else "red"

    @property
    def plot_color_cnr(self) -> str:
        return "green" if self.passed_cnr_constant else "red"

    def as_dict(self) -> dict:
        """Dump important data as a dictionary. Useful when exporting a `results_data` output"""
        return {
            "contrast method": self.contrast_method,
            "visibility": self.visibility,
            "visibility threshold": self.visibility_threshold,
            "passed visibility": bool(self.passed_visibility),
            "contrast": self.contrast,
            "cnr": self.contrast_to_noise,
            "signal to noise": self.signal_to_noise,
        }


class HighContrastDiskROI(DiskROI):
    """A high-contrast disk with a visibility threshold (core/roi.py:411-478)."""

    contrast_threshold: float | None

    @classmethod
    def from_phantom_center(cls, array, angle: float, roi_radius: float, dist_from_center: float, phantom_center,
                            contrast_threshold: float):
        center = cls._get_shifted_center(angle, dist_from_center, phantom_center)
        return cls(array=array, radius=roi_radius, center=center, contrast_threshold=contrast_threshold)

    def __init__(self, array, radius: float, center: Point, contrast_threshold: float):
        super().__init__(array=array, radius=radius, center=center)
        self.contrast_threshold = contrast_threshold

    def __repr__(self):
        return f"High-Contrast Disk; max pixel: {self.max}, min pixel: {self.min}"


class RectangleROI(Rectangle):
    def __init__(self, array: np.ndarray, width: float, height: float, center, rotation: float = 0.0):
        if width < 2:
            raise ValueError(f"The width must be >= 2. Given {width}")
        if height < 2:
            raise ValueError(f"The height must be >= 2. Given {height}")
        super().__init__(width, height, center, rotation=rotation)
        self._array = array
        self._stats = None

    @classmethod
    def from_phantom_center(cls, array, width: float, height: float, angle: float, dist_from_center: float, phantom_center: Point,
                            rotation: float = 0.0):
        """core/roi.py:484-531"""
        y_shift = np.sin(np.deg2rad(angle)) * dist_from_center
        x_shift = np.cos(np.deg2rad(angle)) * dist_from_center
        return cls(array=array, width=width, height=height, center=Point(phantom_center.x + x_shift, phantom_center.y + y_shift),
                   rotation=rotation)

    def _polygon_xy(self) -> np.ndarray:
        """The corner list ``pixels_flat`` hands to skimage.draw.polygon (core/roi.py:646-656), as (x, y) pairs."""
        bl, br, tr, tl = self.bl_corner, self.br_corner, self.tr_corner, self.tl_corner
        return np.array([(bl.x, bl.y - 1), (br.x - 1, br.y - 1), (tr.x - 1, tr.y), (tl.x, tl.y)], dtype=np.float64)

    def _compute(self) -> dict:
        if self._stats is None:
            a = np.asarray(getattr(self._array, "array", self._array))
            if a.dtype not in nat._NP2DT:
                a = a.astype(np.float64)
            out = nat.roi_stats(nat.Context.default(), a, self._polygon_xy()[None])
            self._stats = {k: float(v[0, 0]) for k, v in out.items()}
        return self._stats

    @property
    def pixel_array(self) -> np.ndarray:
        if self.rotation != 0:
            raise ValueError("The pixel array cannot be reshaped into a 2D array when the rotation is not 0.")
        a = getattr(self._array, "array", self._array)
        return a[int(np.round(self.tl_corner.y)): int(np.round(self.bl_corner.y)), int(np.round(self.bl_corner.x)): int(np.round(self.br_corner.x))]

    @property
    def pixel_value(self) -> float:
        return self._compute()["mean"]

    @property
    def mean(self) -> float:
        return self._compute()["mean"]

    @property
    def std(self) -> float:
        return self._compute()["std"]

    @property
    def min(self) -> float:
        return self._compute()["min"]

    @property
    def max(self) -> float:
        return self._compute()["max"]

    def __repr__(self):
        return f"Rectangle ROI @ {self.center}; mean pixel: {self.pixel_value}"
