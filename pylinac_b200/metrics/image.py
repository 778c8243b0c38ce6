"""2-D image metric plug-ins -- mirror of ``pylinac.metrics.image`` (metrics/image.py:38-272, 402-667, 959-983): ``MetricBase``,
``DiskROIMetric`` / ``RectangleROIMetric`` (ROI samplers), ``SizedDiskRegion`` / ``SizedDiskLocator`` (the BB finder) and
``WeightedCentroid``, computed through ``image.compute(metric)``.

The pixel work runs on the device: the disk locator is the threshold sweep / labelling / region-property kernel of the
Winston-Lutz pipeline exposed on its own (``epid_disk_locate``, csrc/wl.cu), the weighted centroid is a device reduction
(``epid_weighted_centroid``, csrc/roi.cu).  Plotting hooks are out of scope.
"""
from __future__ import annotations

import math
import weakref
from abc import ABC, abstractmethod
from typing import Any

import numpy as np

from .. import _native as nat
from ..core.geometry import Point
from ..core.roi import DiskROI, RectangleROI
from .features import DEFAULT_CONDITIONS, conditions_mask


class MetricBase(ABC):
    """metrics/image.py:38-76"""

    unit: str = ""
    image_compatibility = None
    name: str

    def inject_image(self, image) -> None:
        if self.image_compatibility is not None and not isinstance(image, tuple(self.image_compatibility)):
            raise TypeError(f"Image must be one of {self.image_compatibility}")
        self.image = weakref.proxy(image)

    def context_calculate(self) -> Any:
        """Calculate the metric; a metric must not modify the image (hash check, metrics/image.py:61-71)."""
        img_hash = hash(self.image.array.tobytes())
        calculation = self.calculate()
        if hash(self.image.array.tobytes()) != img_hash:
            raise RuntimeError("A metric modified an image. This is not allowed as this could affect other, downstream metrics. "
                               "Change the calculate method to not modify the underlying image.")
        return calculation

    @abstractmethod
    def calculate(self) -> Any:
        ...

    def plot(self, axis, **kwargs) -> None:        # presentation: out of scope
        pass

    def plotly(self, fig, **kwargs) -> None:
        pass

    def additional_plots(self):
        pass


class DiskROIMetric(MetricBase):
    """Samples a disk ROI of the image -> ``DiskROI`` (metrics/image.py:98-177).  ``from_physical`` takes mm; like the reference,
    ``calculate()`` scales the radius and the centre by dpmm IN PLACE every time it runs (:159-161)."""

    roi: DiskROI
    _from_physical: bool = False

    @classmethod
    def from_physical(cls, radius_mm: float, center_mm: Point, name: str = "Disk ROI Metric", edgecolor: str = "b", **kwargs):
        instance = cls(radius_mm, center_mm, name, edgecolor, **kwargs)
        instance._from_physical = True
        return instance

    def __init__(self, radius: float, center: Point, name: str = "Disk ROI Metric", edgecolor: str = "b", **kwargs):
        self.radius = radius
        self.center = center
        self.name = name
        self.edge_color = edgecolor
        self.kwargs = kwargs

    def calculate(self) -> DiskROI:
        if self._from_physical:
            self.radius *= self.image.dpmm
            self.center *= self.image.dpmm
        self.roi = DiskROI(array=self.image.array, center=self.center, radius=self.radius)
        return self.roi


class RectangleROIMetric(MetricBase):
    """Samples a rectangle ROI of the image -> ``RectangleROI`` (metrics/image.py:180-272); ``from_physical`` scales width, height and
    centre by dpmm in place on every ``calculate()`` (:246-250), as the reference does."""

    roi: RectangleROI
    _from_physical: bool = False

    @classmethod
    def from_physical(cls, width_mm: float, height_mm: float, center_mm: Point, name: str = "Rectangle ROI Metric", edgecolor: str = "b",
                      **kwargs):
        instance = cls(width_mm, height_mm, center_mm, name, edgecolor, **kwargs)
        instance._from_physical = True
        return instance

    def __init__(self, width: float, height: float, center: Point, name: str = "Rectangle ROI Metric", edgecolor: str = "b", **kwargs):
        self.height = height
        self.width = width
        self.center = center
        self.name = name
        self.edge_color = edgecolor
        self.kwargs = kwargs

    def calculate(self) -> RectangleROI:
        if self._from_physical:
            self.width *= self.image.dpmm
            self.height *= self.image.dpmm
            self.center *= self.image.dpmm
        self.roi = RectangleROI(array=self.image.array, center=self.center, width=self.width, height=self.height)
        return self.roi


class DiskRegion:
    """The region properties the reference reads from scikit-image's ``RegionProperties`` for a detected disk (sample-window
    coordinates like ``regionprops``): area, area_filled, bbox, area_bbox, centroid, centroid_weighted, perimeter, area_convex,
    solidity -- with the older skimage aliases."""

    def __init__(self, row, k: int):
        self.area = float(row["r_area"][k])
        self.area_filled = self.filled_area = float(row["r_filled_area"][k])
        self.perimeter = float(row["r_perimeter"][k])
        self.area_convex = self.convex_area = float(row["r_convex_area"][k])
        self.solidity = self.area / self.area_convex if self.area_convex else float("nan")
        self.bbox = tuple(int(v) for v in row["r_bbox"][k])
        self.area_bbox = self.bbox_area = float((self.bbox[2] - self.bbox[0]) * (self.bbox[3] - self.bbox[1]))
        self.centroid = (float(row["r_centroid_y"][k]), float(row["r_centroid_x"][k]))
        self.centroid_weighted = self.weighted_centroid = (float(row["r_wcentroid_y"][k]), float(row["r_wcentroid_x"][k]))

    def __repr__(self):
        return f"DiskRegion(area={self.area:.0f}, bbox={self.bbox}, centroid_weighted=({self.centroid_weighted[0]:.2f}, {self.centroid_weighted[1]:.2f}))"


class SizedDiskRegion(MetricBase):
    """metrics/image.py:402-612.  Same constructors (pixels / ``from_physical`` / ``from_center`` / ``from_center_physical``) and the
    same unit bookkeeping as the reference, including that every conversion is applied IN PLACE on each ``calculate()`` call
    (:571-587; ``Point.__mul__`` mutates the expected position, core/geometry.py:190-196)."""

    def __init__(self, expected_position, search_window, radius: float, radius_tolerance: float,
                 detection_conditions=DEFAULT_CONDITIONS, invert: bool = True, name: str = "Disk Region", max_number: int = 1,
                 min_number: int = 1, min_separation_pixels: float = 5):
        self.expected_position = Point(expected_position)
        self.radius = radius
        self.radius_tolerance = radius_tolerance
        self.search_window = search_window
        self.detection_conditions = detection_conditions
        self.name = name
        self.invert = invert
        self.is_from_center = False
        self.is_from_physical = False
        self.max_number = max_number
        self.min_number = min_number
        self.min_separation = min_separation_pixels

    @classmethod
    def from_physical(cls, expected_position_mm, search_window_mm, radius_mm: float, radius_tolerance_mm: float,
                      detection_conditions=DEFAULT_CONDITIONS, invert: bool = True, name="Disk Region", max_number: int = 1,
                      min_number: int = 1, min_separation_mm: float = 5):
        inst = cls(expected_position_mm, search_window_mm, radius_mm, radius_tolerance_mm, detection_conditions, invert, name,
                   max_number, min_number, min_separation_mm)
        inst.is_from_physical = True
        return inst

    @classmethod
    def from_center(cls, expected_position, search_window, radius: float, radius_tolerance: float,
                    detection_conditions=DEFAULT_CONDITIONS, invert: bool = True, name="Disk Region", max_number: int = 1,
                    min_number: int = 1, min_separation_pixels: float = 5):
        inst = cls(expected_position, search_window, radius, radius_tolerance, detection_conditions, invert, name, max_number,
                   min_number, min_separation_pixels)
        inst.is_from_center = True
        return inst

    @classmethod
    def from_center_physical(cls, expected_position_mm, search_window_mm, radius_mm: float, radius_tolerance_mm: float = 0.25,
                             detection_conditions=DEFAULT_CONDITIONS, invert: bool = True, name="Disk Region", max_number: int = 1,
                             min_number: int = 1, min_separation_mm: float = 5):
        inst = cls(expected_position_mm, search_window_mm, radius_mm, radius_tolerance_mm, detection_conditions, invert, name,
                   max_number, min_number, min_separation_mm)
        inst.is_from_physical = True
        inst.is_from_center = True
        return inst

    def _locate(self) -> np.ndarray:
        from ..core import image as _image

        dpmm = self.image.dpmm
        if self.is_from_physical:
            self.expected_position * dpmm                                       # in place (:573)
            self.search_window = np.asarray(self.search_window) * dpmm
        else:
            self.min_separation /= dpmm
            self.radius /= dpmm
            self.radius_tolerance /= dpmm
        if self.is_from_center:
            self.expected_position.x += self.image.shape[1] / 2
            self.expected_position.y += self.image.shape[0] / 2
        p = nat.DiskParams()
        p.dpmm = float(dpmm)
        p.expected_x, p.expected_y = float(self.expected_position.x), float(self.expected_position.y)
        p.window_w, p.window_h = float(self.search_window[0]), float(self.search_window[1])
        p.radius_mm, p.tolerance_mm = float(self.radius), float(self.radius_tolerance)
        p.min_separation_px = float(self.min_separation * dpmm)
        p.invert = 1 if self.invert else 0
        p.max_number = int(self.max_number)
        p.conditions = conditions_mask(self.detection_conditions)
        frame = _image.frame_u16(self.image, "disk locator")
        row = nat.disk_locate(nat.Context.default(), frame, p)[0]
        status = int(row["status"])
        if status == 4:
            raise MemoryError("disk locator: the search window or a candidate region exceeds the device tile (EPID_WL_CAPACITY)")
        n = int(row["n_points"]) if status == 0 else 0
        if n < self.min_number:        # metrics/utils.py:181-185
            raise ValueError(f"Couldn't find the minimum number of disks in the image. Found {n}; required: {self.min_number}")
        return row

    def calculate(self) -> list[DiskRegion]:
        row = self._locate()
        self.x_offset = int(row["left"])
        self.y_offset = int(row["top"])
        self.points = [Point(float(row["x"][k]), float(row["y"][k])) for k in range(int(row["n_points"]))]
        self.boundaries = []           # plot-only outlines (metrics/utils.py:40-63): not produced
        return [DiskRegion(row, k) for k in range(int(row["n_regions"]))]


class SizedDiskLocator(SizedDiskRegion):
    """metrics/image.py:661-667: the weighted centroids of the detected disks as Points (image coordinates)."""

    def calculate(self) -> list[Point]:
        super().calculate()
        return self.points


class WeightedCentroid(MetricBase):
    """metrics/image.py:959-983"""

    def __init__(self, name: str = "Weighted Centroid"):
        self.name = name

    def calculate(self) -> Point:
        arr = np.asarray(self.image.array)
        cx, cy, total = nat.weighted_centroid(nat.Context.default(), arr if arr.dtype in nat._NP2DT else arr.astype(np.float64))
        if total[0] == 0:
            raise ValueError("Image is blank; cannot calculate weighted centroid")
        return Point(float(cx[0]), float(cy[0]))


# ---------------------------------------------------------------------------------------------- whole-frame locators
def _dedupe(total: list[Point], new_points: list[Point], min_separation_px: float) -> list[Point]:
    """metrics/utils.py:14-37: a new point is dropped when it is closer than the separation to any point kept so far (including the
    ones added in this very call: the reference iterates the list it appends to)"""
    for p in new_points:
        if all(p.distance_to(q) >= min_separation_px for q in total):
            total.append(p)
    return total


def _by_threshold(regions: np.ndarray):
    """the accepted regions grouped by threshold, thresholds and labels ascending (the order the reference visits them)"""
    if len(regions) == 0:
        return
    cuts = np.flatnonzero(np.diff(regions["threshold_index"])) + 1
    yield from np.split(regions, cuts)


class GlobalSizedDiskLocator(MetricBase):
    """metrics/image.py:275-354: BBs anywhere in the image.  The threshold sweep, labelling and region analysis of the WHOLE frame
    run on the device (``epid_global_locate``, csrc/locate.cu); the reference's point bookkeeping runs on the returned records."""

    def __init__(self, radius_mm: float, radius_tolerance_mm: float, detection_conditions=None, invert: bool = True, min_number: int = 1,
                 max_number: int | None = None, min_separation_mm: float = 5, name="Global Disk Locator"):
        from .features import is_right_circumference, is_right_size_bb, is_round

        self.radius = radius_mm
        self.radius_tolerance = radius_tolerance_mm
        self.detection_conditions = detection_conditions if detection_conditions is not None else (is_round, is_right_size_bb, is_right_circumference)
        self.name = name
        self.invert = invert
        self.min_number = min_number
        self.max_number = max_number or 1e3
        self.min_separation_mm = min_separation_mm

    def _params(self, dpmm: float, sample_kind: int = 0) -> "nat.LocateParams":
        p = nat.LocateParams()
        p.mode, p.invert, p.sample_kind = 0, int(bool(self.invert)), sample_kind
        p.conditions = conditions_mask(self.detection_conditions)
        p.dpmm = float(dpmm)
        p.radius_mm, p.tolerance_mm = float(self.radius), float(self.radius_tolerance)
        p.bb_size_mm = float(self.radius)           # find_features passes the radius as bb_size (metrics/utils.py:144-150)
        return p

    def _merge(self, regions: np.ndarray, dpmm: float) -> list[Point]:
        total: list[Point] = []
        self.regions = []
        for grp in _by_threshold(regions):
            if len(total) >= self.max_number:
                break
            _dedupe(total, [Point(float(r["wcentroid_x"]), float(r["wcentroid_y"])) for r in grp], self.min_separation_mm * dpmm)
            self.regions = grp
        if len(total) < self.min_number:
            raise ValueError(f"Couldn't find the minimum number of disks in the image. Found {len(total)}; required: {self.min_number}")
        return total

    def calculate(self) -> list[Point]:
        from ..core import image as _image

        dpmm = self.image.dpmm
        frame = _image.frame_u16(self.image, "global disk locator")
        regs = nat.global_locate(nat.Context.default(), frame, self._params(dpmm))[0]
        self.points = self._merge(regs, dpmm)
        self.y_boundaries, self.x_boundaries = [], []       # plot-only outlines: not produced
        return self.points


def locate_disks_batch(frames, dpmm: float, radius_mm: float, radius_tolerance_mm: float, **kwargs) -> list[list[Point]]:
    """GlobalSizedDiskLocator on n uint16 frames [n, H, W] in one device sweep -> one point list per frame ([] where the reference
    would raise for too few disks)."""
    m = GlobalSizedDiskLocator(radius_mm, radius_tolerance_mm, **kwargs)
    out = []
    for regs in nat.global_locate(nat.Context.default(), frames, m._params(dpmm)):
        try:
            out.append(m._merge(regs, dpmm))
        except ValueError:
            out.append([])
    return out


class GlobalSizedFieldLocator(MetricBase):
    """metrics/image.py:727-920: radiation fields anywhere in the image (8-connectivity, clear_border(buffer_size=3), unweighted
    centroids, separation = the largest equivalent diameter of the threshold's fields / dpmm, like the reference)."""

    is_from_physical: bool = False

    def __init__(self, field_width_px: float, field_height_px: float, field_tolerance_px: float, min_number: int = 1,
                 max_number: int | None = None, name: str = "Field Finder", detection_conditions=None):
        from .features import is_right_area_square, is_right_square_perimeter

        self.field_width_mm = field_width_px
        self.field_height_mm = field_height_px
        self.field_tolerance_mm = field_tolerance_px
        self.min_number = min_number
        self.max_number = max_number or 1e6
        self.name = name
        self.detection_conditions = detection_conditions if detection_conditions is not None else (is_right_square_perimeter, is_right_area_square)

    @classmethod
    def from_physical(cls, field_width_mm: float, field_height_mm: float, field_tolerance_mm: float, min_number: int = 1,
                      max_number: int | None = None, name: str = "Field Finder", detection_conditions=None):
        inst = cls(field_width_mm, field_height_mm, field_tolerance_mm, min_number, max_number, name, detection_conditions)
        inst.is_from_physical = True
        return inst

    def _params(self, dpmm: float, sample_kind: int = 0) -> "nat.LocateParams":
        p = nat.LocateParams()
        p.mode, p.invert, p.sample_kind = 1, 0, sample_kind
        p.conditions = conditions_mask(self.detection_conditions)
        p.dpmm = float(dpmm)
        p.field_width_mm, p.field_height_mm, p.field_tolerance_mm = float(self.field_width_mm), float(self.field_height_mm), float(self.field_tolerance_mm)
        return p

    def _merge(self, regions: np.ndarray, dpmm: float) -> list[Point]:
        fields: list[Point] = []
        for grp in _by_threshold(regions):
            if len(fields) >= self.max_number:
                break
            sep = float(grp["equivalent_diameter"].max()) / dpmm          # metrics/image.py:880-884
            _dedupe(fields, [Point(float(r["centroid_x"]), float(r["centroid_y"])) for r in grp], sep)
        if len(fields) < self.min_number:
            raise ValueError(f"Couldn't find the minimum number of fields in the image. Found {len(fields)}; required: {self.min_number}")
        return fields

    def calculate(self, sample_kind: int | None = None) -> list[Point]:
        from ..core import image as _image

        dpmm = self.image.dpmm
        if not self.is_from_physical:          # converted in place on every call, like the reference (:820-823)
            self.field_width_mm /= dpmm
            self.field_height_mm /= dpmm
            self.field_tolerance_mm /= dpmm
        frame = _image.frame_u16(self.image, "global field locator")
        kind = getattr(self.image, "_locator_sample_kind", 0) if sample_kind is None else sample_kind
        regs = nat.global_locate(nat.Context.default(), frame, self._params(dpmm, kind))[0]
        self.fields = self._merge(regs, dpmm)
        self.boundaries = []
        return self.fields


class GlobalFieldLocator(GlobalSizedFieldLocator):
    """metrics/image.py:923-956: fields of any size (the size window is opened to 1e4)."""

    def __init__(self, min_number: int = 1, max_number: int | None = None, name: str = "Field Finder", detection_conditions=None):
        super().__init__(field_width_px=1e4, field_height_px=1e4, field_tolerance_px=1e4, min_number=min_number, max_number=max_number,
                         name=name, detection_conditions=detection_conditions)

    @classmethod
    def from_physical(cls, *args, **kwargs):
        raise NotImplementedError("This method is not implemented for global field-finding. Use the standard initializer instead.")
