"""Generate tests/golden/disk_roi_golden.npz: the UNMODIFIED reference DiskROI / LowContrastDiskROI / HighContrastDiskROI
(core/roi.py:39-479), contrast functions (core/contrast.py), MTF / MomentMTF (core/mtf.py:32-305) and DiskROIMetric /
RectangleROIMetric (metrics/image.py:98-272), stub-imported through oracle/refstub.py, on the seeded frames of disk_roi_cases.py.
skimage.draw.disk is served by tests/golden/skimage_draw.py (restated, parity with scikit-image unpinned), skimage.draw.polygon by
oracle/skimage_shim.py.  Run here:  python -m tests.golden.make_disk_roi_golden

Layout: "<group>/<case>/<quantity>" -> value, or "<group>/<case>/<quantity>!" -> the exception class name the reference raised."""
from __future__ import annotations

import sys
import warnings

import numpy as np

from tests.golden import disk_roi_cases as dc


def _record(store, key, fn, quiet=True):
    try:
        with warnings.catch_warnings():
            if quiet:
                warnings.simplefilter("ignore")
            v = fn()
    except Exception as e:          # the reference's outcome is part of the golden
        store[key + "!"] = np.array(type(e).__name__)
        return None
    store[key] = np.asarray(v)
    return v


def main():
    from oracle import skimage_shim
    from oracle.refstub import import_reference
    from tests.golden import skimage_draw

    import_reference()
    skimage_shim.install()
    skimage_draw.install()
    from pylinac.core import contrast as rc
    from pylinac.core import image as rimage
    from pylinac.core import mtf as rmtf
    from pylinac.core import roi as rroi
    from pylinac.core.geometry import Point
    from pylinac.metrics import image as rmi

    store = {"numpy_version": np.array(np.__version__)}
    raw = dc.raw_frame()
    for kind in ("f64", "f32"):        # the case module's ground / normalize is the reference's
        img = rimage.ArrayImage(raw.astype(np.float32) if kind == "f32" else raw.copy(), dpi=dc.DPI)
        img.ground()
        img.normalize()
        a = dc.frame(kind)
        assert img.array.dtype == a.dtype and np.array_equal(img.array, a), kind

    parity = set()
    for kind in dc.KINDS:
        a = dc.frame(kind)
        for name, (x, y, r) in dc.DISKS.items():
            k = f"{kind}/{name}"
            roi = rroi.LowContrastDiskROI(a, r, Point(x, y))
            px = _record(store, f"{k}/count", lambda: len(roi.circle_mask()))
            if px is not None and name in dc.SMALL_DISKS:
                store[f"{k}/pixel_values"] = np.asarray(roi.pixel_values)
            if px is not None:
                parity.add(px % 2)
            for q in ("pixel_value", "mean", "std", "min", "max"):
                _record(store, f"{k}/{q}", lambda: getattr(roi, q))
            _record(store, f"{k}/percentile", lambda: [roi.percentile(p) for p in dc.PERCENTILES])
            m = _record(store, f"{k}/masked_array", lambda: roi.masked_array()) if name in dc.SMALL_DISKS else None
            if m is not None:
                # stored sparsely: the fill value np.full(shape, np.nan, dtype) gives (0 after numpy's invalid cast for an integer
                # image), the flat indices that differ from it and their values
                del store[f"{k}/masked_array"]
                with warnings.catch_warnings():
                    warnings.simplefilter("ignore")
                    fill = np.full((), np.nan, dtype=m.dtype)
                idx = np.flatnonzero(~np.isnan(m)) if np.isnan(fill) else np.flatnonzero(m != fill)
                store[f"{k}/masked_fill"] = fill
                store[f"{k}/masked_idx"] = idx
                store[f"{k}/masked_vals"] = m.ravel()[idx]
            _record(store, f"{k}/as_dict", lambda: [float(v) for v in rroi.DiskROI(a, r, Point(x, y)).as_dict().values()])
        _record(store, f"{kind}/percentile_out_of_range", lambda: rroi.LowContrastDiskROI(a, 5, Point(100, 100)).percentile(100.5))
    assert parity == {0, 1}, "the disk set must have odd and even pixel counts"

    # LowContrastDiskROI contrast / visibility / pass-fail on the normalised float64 frame, every method, with and without reference
    a = dc.frame("f64")
    props = ("contrast", "visibility", "contrast_to_noise", "signal_to_noise", "michelson", "weber", "rms", "ratio", "cnr_constant",
             "contrast_constant", "passed", "passed_visibility", "passed_contrast_constant", "passed_cnr_constant")
    for name, ref in dc.LOW_CONTRAST:
        x, y, r = dc.DISKS[name]
        for method in dc.CONTRAST_METHODS:
            k = f"low/{name}/{method}"
            roi = rroi.LowContrastDiskROI(a, r, Point(x, y), contrast_threshold=0.05, contrast_reference=ref, cnr_threshold=3.0,
                                          contrast_method=method, visibility_threshold=0.2)
            store[f"{k}/inputs"] = np.array([roi.pixel_value, roi.std, r, np.nan if ref is None else ref])
            for p in props:
                _record(store, f"{k}/{p}", lambda: getattr(roi, p))
            _record(store, f"{k}/as_dict", lambda: [str(v) for v in roi.as_dict().values()])
            # the module-level functions on the same inputs
            arr = np.array((roi.pixel_value, ref))
            _record(store, f"{k}/fn_contrast", lambda: rc.contrast(arr, method))
            _record(store, f"{k}/fn_visibility", lambda: rc.visibility(arr, r, roi.std, method))
            _record(store, f"{k}/fn_contrast_upper", lambda: rc.contrast(arr, method.upper()))
    for k, arr in {"pair": np.array([0.62, 0.48]), "spread": np.array([0.1, 0.4, 0.35, 0.9]), "negative": np.array([-0.1, 0.5]),
                   "above_one": np.array([0.5, 1.5]), "nan": np.array([0.3, np.nan, 0.7])}.items():
        store[f"fn/{k}/array"] = arr
        _record(store, f"fn/{k}/michelson", lambda: rc.michelson(arr))
        _record(store, f"fn/{k}/rms", lambda: rc.rms(arr))
        for method in dc.CONTRAST_METHODS:
            _record(store, f"fn/{k}/contrast/{method}", lambda: rc.contrast(arr, method))
        _record(store, f"fn/{k}/contrast/unknown", lambda: rc.contrast(arr, "nope"))
        _record(store, f"fn/{k}/weber", lambda: rc.weber(arr[0], arr[-1]))
        _record(store, f"fn/{k}/ratio", lambda: rc.ratio(arr[0], arr[-1]))
        _record(store, f"fn/{k}/difference", lambda: rc.difference(arr[0], arr[-1]))

    # MTF / MomentMTF from high-contrast disk sets (uint16 frame)
    u = dc.frame("u16")
    for name, (spacings, centres, r) in dc.MTF_SETS.items():
        k = f"mtf/{name}"
        disks = [rroi.HighContrastDiskROI(u, r, Point(*c), contrast_threshold=0.5) for c in centres]
        store[f"{k}/max"] = np.array([d.max for d in disks])
        store[f"{k}/min"] = np.array([d.min for d in disks])
        store[f"{k}/mean"] = np.array([d.mean for d in disks])
        store[f"{k}/std"] = np.array([d.std for d in disks])
        with warnings.catch_warnings(record=True) as wl:
            warnings.simplefilter("always")
            mtf = rmtf.MTF.from_high_contrast_diskset(spacings, disks)
        store[f"{k}/warn_monotonic"] = np.array(sum("monotonically" in str(w.message) for w in wl))
        store[f"{k}/norm_mtfs"] = np.array([list(mtf.norm_mtfs.keys()), list(mtf.norm_mtfs.values())])
        store[f"{k}/mtfs"] = np.array(list(mtf.mtfs.values()))
        for x in dc.MTF_RESOLUTIONS:
            with warnings.catch_warnings(record=True) as wl:
                warnings.simplefilter("always")
                _record(store, f"{k}/rr/{x}", lambda: mtf.relative_resolution(x), quiet=False)
            store[f"{k}/rr/{x}/warn"] = np.array(sum("extrapolation" in str(w.message) for w in wl))
        mm = _record(store, f"{k}/moment", lambda: rmtf.MomentMTF.from_high_contrast_diskset(spacings, disks))
        if mm is not None:
            del store[f"{k}/moment"]
            store[f"{k}/moment_mtfs"] = np.array(list(mm.mtfs.values()))
            store[f"{k}/moment_fwhms"] = np.array(list(mm.fwhms.values()))
    _record(store, "mtf/unequal", lambda: rmtf.MTF([0.1, 0.2], [1.0, 0.9, 0.8], [0.1, 0.2]))
    _record(store, "mtf/too_few", lambda: rmtf.MTF([0.1], [1.0], [0.1]))
    _record(store, "mtf/moments_domain", lambda: rmtf.moments_mtf(100.0, 5.0))

    # metrics through compute (float64 frame), each computed twice
    for name, (cls_name, physical, kw) in dc.METRICS.items():
        k = f"metric/{name}"
        img = rimage.ArrayImage(dc.frame("f64"), dpi=dc.DPI)
        kw = {key: (Point(*v) if isinstance(v, tuple) else v) for key, v in kw.items()}
        cls = getattr(rmi, cls_name)
        metric = cls.from_physical(**kw) if physical else cls(**kw)
        for run in range(2):
            roi = img.compute(metrics=metric)
            qs = ("pixel_value", "mean", "std", "min", "max") if cls_name == "DiskROIMetric" else ("mean", "std", "min", "max")
            store[f"{k}/{run}/stats"] = np.array([float(getattr(roi, q)) for q in qs])
            store[f"{k}/{run}/center"] = np.array([metric.center.x, metric.center.y])
            store[f"{k}/{run}/size"] = np.array([metric.radius] if cls_name == "DiskROIMetric" else [metric.width, metric.height])
    np.savez_compressed("tests/golden/disk_roi_golden.npz", **store)
    print(len(store), "entries")


if __name__ == "__main__":
    sys.exit(main())
