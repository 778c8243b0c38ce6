"""CPU: the host side of the disk-ROI layer against tests/golden/disk_roi_golden.npz (the unmodified reference, see
tests/golden/make_disk_roi_golden.py): the contrast functions, the LowContrastDiskROI contrast / visibility / pass-fail properties on
the reference's own statistics, MTF / MomentMTF / relative_resolution, argument errors, and the restated skimage.draw.disk of
tests/golden/skimage_draw.py against a brute-force evaluation of its definition.  The pixel-set rule itself is restated from
scikit-image (not installed here), so parity with the real library is unpinned; everything downstream of the pixel set is pinned."""
import math
import os
import warnings

import numpy as np
import pytest

from pylinac_b200.core import contrast as ct
from pylinac_b200.core import mtf as mt
from pylinac_b200.core.geometry import Point
from pylinac_b200.core.roi import DiskROI, HighContrastDiskROI, LowContrastDiskROI, bbox_center
from tests.golden import disk_roi_cases as dc
from tests.golden import skimage_draw

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "disk_roi_golden.npz"))


def check(key, fn, exact=True, quiet=True):
    """Compare fn() with the golden value of key, or the exception class the reference raised."""
    if key + "!" in G.files:
        with pytest.raises(Exception) as ei:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                fn()
        assert type(ei.value).__name__ == str(G[key + "!"]), (key, ei.value)
        return
    with warnings.catch_warnings():
        if quiet:
            warnings.simplefilter("ignore")
        v = fn()
    want = G[key]
    if want.dtype.kind in "US":
        assert np.array_equal(np.asarray(v).astype(str), want), (key, v, want)
    elif exact:
        np.testing.assert_array_equal(np.asarray(v, dtype=want.dtype), want, err_msg=key)
    else:
        np.testing.assert_allclose(np.asarray(v, dtype=float), want, rtol=1e-13, atol=0, err_msg=key)


@pytest.mark.parametrize("k", ["pair", "spread", "negative", "above_one", "nan"])
def test_contrast_functions(k):
    arr = G[f"fn/{k}/array"]
    check(f"fn/{k}/michelson", lambda: ct.michelson(arr))
    check(f"fn/{k}/rms", lambda: ct.rms(arr))
    for method in dc.CONTRAST_METHODS:
        check(f"fn/{k}/contrast/{method}", lambda: ct.contrast(arr, method))
    check(f"fn/{k}/contrast/unknown", lambda: ct.contrast(arr, "nope"))
    check(f"fn/{k}/weber", lambda: ct.weber(arr[0], arr[-1]))
    check(f"fn/{k}/ratio", lambda: ct.ratio(arr[0], arr[-1]))
    check(f"fn/{k}/difference", lambda: ct.difference(arr[0], arr[-1]))


LOW_PROPS = ("contrast", "visibility", "contrast_to_noise", "signal_to_noise", "michelson", "weber", "rms", "ratio", "cnr_constant",
             "contrast_constant", "passed", "passed_visibility", "passed_contrast_constant", "passed_cnr_constant")


@pytest.mark.parametrize("name,ref", dc.LOW_CONTRAST)
@pytest.mark.parametrize("method", dc.CONTRAST_METHODS)
def test_low_contrast_properties_on_reference_statistics(name, ref, method):
    """The property logic on the reference's median and std (injected as the ROI's cached statistics: no device needed)."""
    k = f"low/{name}/{method}"
    pv, std, r, _ = G[f"{k}/inputs"]
    x, y, _ = dc.DISKS[name]
    roi = LowContrastDiskROI(np.zeros(dc.SHAPE), r, Point(x, y), contrast_threshold=0.05, contrast_reference=ref, cnr_threshold=3.0,
                             contrast_method=method, visibility_threshold=0.2)
    roi._stats = {"count": 1.0, "median": float(pv), "std": float(std)}
    for p in LOW_PROPS:
        check(f"{k}/{p}", lambda: getattr(roi, p))
    check(f"{k}/as_dict", lambda: [str(v) for v in roi.as_dict().values()])
    arr = np.array((float(pv), ref))
    check(f"{k}/fn_contrast", lambda: ct.contrast(arr, method))
    check(f"{k}/fn_visibility", lambda: ct.visibility(arr, r, float(std), method))
    check(f"{k}/fn_contrast_upper", lambda: ct.contrast(arr, method.upper()))


@pytest.mark.parametrize("name", sorted(dc.MTF_SETS))
def test_mtf_and_moment_mtf(name):
    k = f"mtf/{name}"
    spacings = dc.MTF_SETS[name][0]
    with warnings.catch_warnings(record=True) as wl:
        warnings.simplefilter("always")
        m = mt.MTF(spacings, list(G[f"{k}/max"]), list(G[f"{k}/min"]))
    assert sum("monotonically" in str(w.message) for w in wl) == int(G[f"{k}/warn_monotonic"])
    np.testing.assert_array_equal(np.array([list(m.norm_mtfs.keys()), list(m.norm_mtfs.values())]), G[f"{k}/norm_mtfs"])
    np.testing.assert_array_equal(np.array(list(m.mtfs.values())), G[f"{k}/mtfs"])
    for x in dc.MTF_RESOLUTIONS:
        with warnings.catch_warnings(record=True) as wl:
            warnings.simplefilter("always")
            check(f"{k}/rr/{x}", lambda: m.relative_resolution(x), quiet=False)
        assert sum("extrapolation" in str(w.message) for w in wl) == int(G[f"{k}/rr/{x}/warn"]), x
    mm = mt.MomentMTF(spacings, list(G[f"{k}/mean"]), list(G[f"{k}/std"]))
    np.testing.assert_array_equal(np.array(list(mm.mtfs.values())), G[f"{k}/moment_mtfs"])
    np.testing.assert_array_equal(np.array(list(mm.fwhms.values())), G[f"{k}/moment_fwhms"])
    assert issubclass(mt.PeakValleyMTF, mt.MTF)


def test_mtf_argument_errors():
    check("mtf/unequal", lambda: mt.MTF([0.1, 0.2], [1.0, 0.9, 0.8], [0.1, 0.2]))
    check("mtf/too_few", lambda: mt.MTF([0.1], [1.0], [0.1]))
    check("mtf/moments_domain", lambda: mt.moments_mtf(100.0, 5.0))
    m = mt.MTF([0.1, 0.2, 0.3], [1.0, 0.9, 0.8], [0.1, 0.3, 0.5])
    for bad in (-1, 100.5):
        with pytest.raises(ValueError):
            m.relative_resolution(bad)


def test_interp1d_restatement_matches_scipy():
    """relative_resolution's numpy restatement of interp1d(fill_value="extrapolate") against scipy itself (tests may use scipy)."""
    from scipy.interpolate import interp1d

    rng = np.random.default_rng(7)
    for _ in range(50):
        n = int(rng.integers(2, 9))
        x = rng.uniform(0, 1, n)
        y = np.sort(rng.uniform(0.05, 1.5, n))
        for xn in (-0.3, 0.0, 0.2, 0.5, 0.9, 1.0, 1.7, float(x[0])):
            assert mt._interp1d_extrapolate(x, y, xn) == interp1d(x, y, fill_value="extrapolate")(xn)


def test_constructors_and_geometry():
    a = np.zeros((50, 60), np.uint16)
    d = DiskROI.from_phantom_center(a, angle=90, roi_radius=4, dist_from_center=10, phantom_center=Point(30, 25))
    assert (d.center.x, d.center.y, d.radius, d.diameter) == (30 + np.cos(np.pi / 2) * 10, 35.0, 4, 8)
    lo = LowContrastDiskROI.from_phantom_center(a, 0, 3, 5, Point(10, 10), contrast_threshold=0.1, contrast_reference=0.5,
                                                cnr_threshold=2, contrast_method=ct.Contrast.WEBER, visibility_threshold=0.3)
    assert (lo.center.x, lo.center.y, lo.contrast_method, lo.visibility_threshold, lo.cnr_threshold) == (15, 10, "Weber", 0.3, 2)
    hi = HighContrastDiskROI.from_phantom_center(a, 180, 2, 4, Point(20, 20), contrast_threshold=0.4)
    assert hi.contrast_threshold == 0.4 and math.isclose(hi.center.x, 16)
    with pytest.raises(TypeError):
        DiskROI(a, 3, "centre")
    with pytest.raises(TypeError):
        HighContrastDiskROI(a, 3, Point(1, 1))           # contrast_threshold is required
    assert ct.Contrast.options() == ["Michelson", "Weber", "Ratio", "Root Mean Square", "Difference"]

    class Region:
        bbox = (10, 20, 30, 50)

    c = bbox_center(Region())
    assert (c.x, c.y) == (35.0, 20.0)


@pytest.mark.parametrize("clip", [False, True])
def test_shim_disk_against_brute_force(clip):
    """skimage_draw.disk against its own definition evaluated pixel by pixel over a padded window: ((i - r_org) / r)**2 +
    ((j - c_org) / r)**2 < 1 relative to the box corner, row-major order, clipped only with a shape."""
    rng = np.random.default_rng(11)
    shape = (40, 50)
    cases = [(10.5, 12.5, 0.5), (20.0, 25.0, 5.0), (7.25, 3.75, 4.5), (-1.5, 2.0, 3.0), (38.2, 48.9, 6.3)]
    cases += [tuple(rng.uniform(-5, 45, 2)) + (float(rng.uniform(0.3, 12)),) for _ in range(40)]
    for cy, cx, r in cases:
        rr, cc = skimage_draw.disk((cy, cx), r, shape=shape if clip else None)
        r0, c0 = math.ceil(cy - r), math.ceil(cx - r)
        r1, c1 = math.floor(cy + r), math.floor(cx + r)
        if clip:
            r0, c0, r1, c1 = max(r0, 0), max(c0, 0), min(r1, shape[0] - 1), min(c1, shape[1] - 1)
        want = [(i, j) for i in range(r0, r1 + 1) for j in range(c0, c1 + 1)
                if (((i - r0) - (cy - r0)) / r) ** 2 + (((j - c0) - (cx - c0)) / r) ** 2 < 1]
        assert list(zip(rr.tolist(), cc.tolist())) == want, (cy, cx, r)
