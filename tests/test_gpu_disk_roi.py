"""GPU: DiskROI / LowContrastDiskROI / HighContrastDiskROI, sample_disks_batch, MTF from disk sets and the ROI metrics against
tests/golden/disk_roi_golden.npz (the unmodified reference on the seeded frames of tests/golden/disk_roi_cases.py).

The reference's pixel set comes from skimage.draw.disk, restated in tests/golden/skimage_draw.py because scikit-image is not
installed where the goldens are made: parity with the real library is unpinned at that boundary.  Everything downstream of the pixel
set is pinned here: statistics, pixel order, wrap-around over the top / left edges, IndexError over the bottom / right edges, the
empty-disk outcomes, the disk too large to stage in shared memory, contrast and MTF.

Tolerances: order statistics (median, percentiles, min, max) exact for every dtype; 16-bit frames: count / mean exact, std 1e-12
relative; float64 frames: mean / std 1e-12; float32 frames: mean / std 1e-6 (numpy sums float32 in float32)."""
import os
import warnings

import numpy as np
import pytest

from pylinac_b200 import _native as nat
from pylinac_b200.core import mtf as mt
from pylinac_b200.core.geometry import Point
from pylinac_b200.core.image import ArrayImage
from pylinac_b200.core.roi import DiskROI, HighContrastDiskROI, LowContrastDiskROI, sample_disks_batch
from pylinac_b200.metrics import image as mi
from tests.golden import disk_roi_cases as dc

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "disk_roi_golden.npz"))
FRAMES = {k: dc.frame(k) for k in dc.KINDS}
MOMENT_RTOL = {"u16": 1e-12, "f64": 1e-12, "f32": 1e-6}


def outcome(key, fn, rtol=0.0):
    """fn() against the golden value of key (rtol 0 = exact), or the exception class the reference raised."""
    if key + "!" in G.files:
        with pytest.raises(Exception) as ei:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                fn()
        assert type(ei.value).__name__ == str(G[key + "!"]), (key, repr(ei.value))
        return
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        v = np.asarray(fn())
    want = G[key]
    if want.dtype.kind in "US":
        assert np.array_equal(v.astype(str), want), (key, v, want)
    elif rtol == 0 or want.dtype.kind == "b":
        np.testing.assert_array_equal(v, want, err_msg=key)
    else:
        np.testing.assert_allclose(v.astype(float), want, rtol=rtol, atol=0, err_msg=key)


@pytest.mark.parametrize("name", sorted(dc.DISKS))
@pytest.mark.parametrize("kind", dc.KINDS)
def test_disk_statistics_match_reference(kind, name):
    x, y, r = dc.DISKS[name]
    roi = LowContrastDiskROI(FRAMES[kind], r, Point(x, y))
    k = f"{kind}/{name}"
    mrt = MOMENT_RTOL[kind]
    outcome(f"{k}/count", lambda: len(roi.circle_mask()))
    outcome(f"{k}/pixel_value", lambda: roi.pixel_value)
    outcome(f"{k}/min", lambda: roi.min)
    outcome(f"{k}/max", lambda: roi.max)
    outcome(f"{k}/mean", lambda: roi.mean, 0.0 if kind == "u16" else mrt)
    outcome(f"{k}/std", lambda: roi.std, mrt)
    outcome(f"{k}/percentile", lambda: [roi.percentile(p) for p in dc.PERCENTILES])
    outcome(f"{k}/as_dict", lambda: [float(v) for v in DiskROI(FRAMES[kind], r, Point(x, y)).as_dict().values()], mrt)
    if f"{k}/pixel_values" in G.files:          # values and order, wrap-around included
        pv = roi.pixel_values
        assert pv.dtype == G[f"{k}/pixel_values"].dtype
        np.testing.assert_array_equal(pv, G[f"{k}/pixel_values"])
    if f"{k}/masked_idx" in G.files:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            m = roi.masked_array()
        want = np.full(m.shape, G[f"{k}/masked_fill"], dtype=m.dtype)
        want.ravel()[G[f"{k}/masked_idx"]] = G[f"{k}/masked_vals"]
        np.testing.assert_array_equal(m, want)


@pytest.mark.parametrize("kind", dc.KINDS)
def test_percentile_range_error(kind):
    outcome(f"{kind}/percentile_out_of_range", lambda: LowContrastDiskROI(FRAMES[kind], 5, Point(100, 100)).percentile(100.5))


@pytest.mark.parametrize("name,ref", dc.LOW_CONTRAST)
@pytest.mark.parametrize("method", dc.CONTRAST_METHODS)
def test_low_contrast_properties_on_device_statistics(name, ref, method):
    x, y, r = dc.DISKS[name]
    k = f"low/{name}/{method}"
    roi = LowContrastDiskROI(FRAMES["f64"], r, Point(x, y), contrast_threshold=0.05, contrast_reference=ref, cnr_threshold=3.0,
                             contrast_method=method, visibility_threshold=0.2)
    for p in ("contrast", "visibility", "contrast_to_noise", "signal_to_noise", "michelson", "weber", "rms", "ratio", "cnr_constant",
              "contrast_constant", "passed", "passed_visibility", "passed_contrast_constant", "passed_cnr_constant"):
        outcome(f"{k}/{p}", lambda: getattr(roi, p), 1e-11)


@pytest.mark.parametrize("name", sorted(dc.MTF_SETS))
def test_mtf_from_high_contrast_diskset(name):
    spacings, centres, r = dc.MTF_SETS[name]
    k = f"mtf/{name}"
    disks = [HighContrastDiskROI(FRAMES["u16"], r, Point(*c), contrast_threshold=0.5) for c in centres]
    with warnings.catch_warnings(record=True) as wl:
        warnings.simplefilter("always")
        m = mt.MTF.from_high_contrast_diskset(spacings, disks)
    assert sum("monotonically" in str(w.message) for w in wl) == int(G[f"{k}/warn_monotonic"])
    np.testing.assert_array_equal(np.array([list(m.norm_mtfs.keys()), list(m.norm_mtfs.values())]), G[f"{k}/norm_mtfs"])
    for x in dc.MTF_RESOLUTIONS:
        with warnings.catch_warnings(record=True) as wl:
            warnings.simplefilter("always")
            assert m.relative_resolution(x) == float(G[f"{k}/rr/{x}"])
        assert sum("extrapolation" in str(w.message) for w in wl) == int(G[f"{k}/rr/{x}/warn"])
    mm = mt.MomentMTF.from_high_contrast_diskset(spacings, disks)
    np.testing.assert_allclose(list(mm.mtfs.values()), G[f"{k}/moment_mtfs"], rtol=1e-11)
    np.testing.assert_allclose(list(mm.fwhms.values()), G[f"{k}/moment_fwhms"], rtol=1e-11)
    assert "High-Contrast Disk" in repr(disks[0])


@pytest.mark.parametrize("name", sorted(dc.METRICS))
def test_roi_metrics_through_compute(name):
    cls_name, physical, kw = dc.METRICS[name]
    img = ArrayImage(FRAMES["f64"], dpi=dc.DPI)
    kw = {key: (Point(*v) if isinstance(v, tuple) else v) for key, v in kw.items()}
    cls = getattr(mi, cls_name)
    metric = cls.from_physical(**kw) if physical else cls(**kw)
    for run in range(2):          # from_physical scales in place on every calculate(), as the reference
        roi = img.compute(metrics=metric)
        k = f"metric/{name}/{run}"
        qs = ("pixel_value", "mean", "std", "min", "max") if cls_name == "DiskROIMetric" else ("mean", "std", "min", "max")
        np.testing.assert_allclose([float(getattr(roi, q)) for q in qs], G[f"{k}/stats"], rtol=1e-10, atol=0)
        assert [metric.center.x, metric.center.y] == list(G[f"{k}/center"])
        size = [metric.radius] if cls_name == "DiskROIMetric" else [metric.width, metric.height]
        assert size == list(G[f"{k}/size"])
        if cls_name == "DiskROIMetric":
            assert roi.pixel_value == float(G[f"{k}/stats"][0]) and roi.min == float(G[f"{k}/stats"][3])


def _batch_layout():
    rng = np.random.default_rng(99)
    centres, radii = [], []
    for i in range(20):
        r = float(rng.uniform(3, 60))
        if i < 3:           # over the top / left edges: the wrapped rows / columns
            centres.append((float(rng.uniform(-2, 8)) if i != 1 else 500.0, float(rng.uniform(-2, 8)) if i != 0 else 400.0))
        else:
            centres.append((float(rng.uniform(r + 1, 1023 - r)), float(rng.uniform(r + 1, 1023 - r))))
        radii.append(r)
    return centres, radii


def test_sample_disks_batch_matches_per_object_path_and_numpy():
    rng = np.random.default_rng(5)
    frames = rng.normal(20000, 900, (64, 1024, 1024)).clip(0, 65535).astype(np.uint16)
    centres, radii = _batch_layout()
    pcts = (0, 2.5, 50, 97.5, 100)
    ctx = nat.Context.default()
    b = nat.Batch.upload(ctx, frames)
    try:
        out = sample_disks_batch(b, centres, radii, pcts)
    finally:
        b.free()
    assert out["count"].shape == (64, 20) and out["percentile"].shape == (64, 20, 5)
    for f in range(64):
        for d, (c, r) in enumerate(zip(centres, radii)):
            roi = LowContrastDiskROI(frames[f], r, Point(*c))
            got = [roi.pixel_value, roi.mean, roi.std, roi.min, roi.max]
            assert got == [out[q][f, d] for q in ("median", "mean", "std", "min", "max")], (f, d)
            if f % 16 == 0:
                assert [roi.percentile(p) for p in pcts] == list(out["percentile"][f, d]), (f, d)
                v = nat.disk_roi_pixels(ctx, frames[f], 0, c, r)
                assert len(v) == out["count"][f, d]
                assert float(np.median(v)) == out["median"][f, d]
                assert float(np.mean(v)) == out["mean"][f, d]
                assert float(np.min(v)) == out["min"][f, d] and float(np.max(v)) == out["max"][f, d]
                assert [float(np.percentile(v, p)) for p in pcts] == list(out["percentile"][f, d])
                np.testing.assert_allclose(out["std"][f, d], np.std(v), rtol=1e-12)


def test_batch_errors_and_empty():
    a = FRAMES["u16"]
    with pytest.raises(IndexError):
        sample_disks_batch(a, [(100, 100), dc.DISKS["oob_bottom"][:2]], [5, dc.DISKS["oob_bottom"][2]])
    out = sample_disks_batch(a, [dc.DISKS["empty"][:2]], [dc.DISKS["empty"][2]])
    assert out["count"][0, 0] == 0 and np.isnan(out["mean"][0, 0]) and np.isnan(out["median"][0, 0])
    with pytest.raises(ValueError):
        sample_disks_batch(a, [(100, 100)], [5], [101])
    with pytest.raises(ValueError):
        sample_disks_batch(a, [(100, 100)], [5], list(range(nat.DISK_MAX_PCT + 1)))
    with pytest.raises(ValueError):
        sample_disks_batch(a, [(np.nan, 100)], [5])
    with pytest.raises(IndexError):
        nat.disk_roi_pixels(nat.Context.default(), a, 0, dc.DISKS["oob_right"][:2], dc.DISKS["oob_right"][2])
    # clipped pixel set (masked_array) of a disk over the bottom edge: in range, no error
    v, rr, cc = nat.disk_roi_pixels(nat.Context.default(), a, 0, dc.DISKS["oob_bottom"][:2], dc.DISKS["oob_bottom"][2], clip=True,
                                    indices=True)
    assert rr.max() == a.shape[0] - 1 and np.array_equal(v, a[rr, cc])


def test_nan_pixels_make_every_statistic_nan():
    a = FRAMES["f64"].copy()
    x, y, r = dc.DISKS["qc3"]
    a[int(y), int(x)] = np.nan
    roi = LowContrastDiskROI(a, r, Point(x, y))
    v = roi.pixel_values
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for got, want in ((roi.pixel_value, np.median(v)), (roi.mean, np.mean(v)), (roi.std, np.std(v)), (roi.min, np.min(v)),
                          (roi.max, np.max(v)), (roi.percentile(50), np.percentile(v, 50))):
            assert np.isnan(got) and np.isnan(want)
