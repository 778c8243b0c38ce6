"""CPU: the set-level host math of the multi-target Winston-Lutz (BBFieldMatch vectors, BB3D positions, align_points 6-DoF shift;
pylinac_b200/winston_lutz_mtmf.py) against goldens of the UNMODIFIED reference (tests/golden/make_mtmf_golden.py), with the per-image
points taken from the golden file (tests/test_gpu_mtmf.py runs the images through CUDA)."""
import numpy as np
import pytest

from pylinac_b200 import winston_lutz_mtmf as mt
from pylinac_b200.core.geometry import Point
from tests.golden.mtmf_cases import SETS

GOLD = np.load("tests/golden/mtmf_golden.npz")


def build(name):
    arr, _, axes = SETS[name]
    cfgs = tuple(mt.BBConfig(name=n, offset_left_mm=l, offset_up_mm=u, offset_in_mm=i, bb_size_mm=d, rad_size_mm=r) for n, l, u, i, d, r in arr)
    bb, fld, ep = GOLD[f"{name}/bb_px"], GOLD[f"{name}/field_px"], GOLD[f"{name}/epid_px"]
    st = mt.WinstonLutzMultiTargetMultiField.__new__(mt.WinstonLutzMultiTargetMultiField)
    st.images = []
    for k, (g, c, p) in enumerate(axes):
        im = mt.WinstonLutzMultiTargetMultiFieldImage.__new__(mt.WinstonLutzMultiTargetMultiFieldImage)
        im.gantry_angle, im.collimator_angle, im.couch_angle, im.dpmm, im.sad = float(g), float(c), float(p), 2.56, 1000.0
        im.arrangement_matches = {cfg.name: mt.BBFieldMatch(epid=Point(*ep[k]), field=Point(*fld[k, j]), bb=Point(*bb[k, j]), dpmm=2.56,
                                                            gantry_angle=float(g), couch_angle=float(p), sad=1000.0)
                                  for j, cfg in enumerate(cfgs)}
        st.images.append(im)
    st.bb_arrangement = cfgs
    st.machine_scale = mt.MachineScale.IEC61217
    st.bbs = [mt.BB3D(cfg, [im.arrangement_matches[cfg.name] for im in st.images], st.machine_scale) for cfg in cfgs]
    st._is_analyzed = True
    return st


def check(st, name, tol):
    np.testing.assert_allclose([[b.measured_bb_position.x, b.measured_bb_position.y, b.measured_bb_position.z] for b in st.bbs],
                               GOLD[f"{name}/measured_bb"], rtol=0, atol=tol)
    np.testing.assert_allclose([[b.measured_field_position.x, b.measured_field_position.y, b.measured_field_position.z] for b in st.bbs],
                               GOLD[f"{name}/measured_field"], rtol=0, atol=tol)
    t, yaw, pitch, roll = st.bb_shift_vector
    np.testing.assert_allclose([t.x, t.y, t.z, yaw, pitch, roll], GOLD[f"{name}/shift"], rtol=0, atol=max(tol, 1e-9) * 100)
    rd = st.results_data()
    np.testing.assert_allclose(rd.max_2d_field_to_bb_mm, GOLD[f"{name}/max_2d"], rtol=0, atol=tol)
    np.testing.assert_allclose(rd.mean_2d_field_to_bb_mm, GOLD[f"{name}/mean_2d"], rtol=0, atol=tol)
    np.testing.assert_allclose(rd.median_2d_field_to_bb_mm, GOLD[f"{name}/median_2d"], rtol=0, atol=tol)
    np.testing.assert_allclose([rd.bb_maxes[n] for n in GOLD[f"{name}/names"]], GOLD[f"{name}/bb_maxes"], rtol=0, atol=tol)


@pytest.mark.parametrize("name", list(SETS))
def test_mtmf_set_level_matches_reference(name):
    st = build(name)
    check(st, name, 1e-10)
    assert st.bb_shift_instructions() == str(GOLD[f"{name}/instructions"])


def test_align_points_recovers_a_known_rigid_motion():
    rng = np.random.default_rng(5)
    pts = rng.uniform(-50, 50, size=(6, 3))
    yaw, pitch, roll = 1.5, -0.7, 2.2
    R = mt._rot("z", np.radians(yaw)) @ mt._rot("x", np.radians(pitch)) @ mt._rot("y", np.radians(roll))
    moved = pts @ R.T + np.array([0.4, -1.1, 2.0])
    t, y, p, r = mt.align_points([Point(*q) for q in pts], [Point(*q) for q in moved])
    np.testing.assert_allclose([y, p, r], [yaw, pitch, roll], atol=1e-9)
    np.testing.assert_allclose([t.x, t.y, t.z], [0.4, -1.1, 2.0], atol=1e-9)


def test_align_points_other_axes_orders_follow_the_reference_call():
    """winston_lutz.py:3592-3605, 3655-3658: any order of 'roll', 'pitch', 'yaw' is turned into an extrinsic euler string and the three
    angles of Rotation.as_euler are unpacked POSITIONALLY as (roll, pitch, yaw).  The default order also goes through scipy here and
    must equal the closed form the module uses for it; the unmodified reference's results are stored in tests/golden/fresh_golden.npz
    (tests/golden/make_fresh_golden.py)."""
    from scipy.spatial.transform import Rotation

    from tests.golden import fresh_cases as fc

    pts, moved = fc.align_points_inputs()
    R = Rotation.from_euler("yxz", [2.2, -0.7, 1.5], degrees=True).as_matrix()
    mp_, ip_ = [Point(*q) for q in pts], [Point(*q) for q in moved]
    t0, y0, p0, r0 = mt.align_points(mp_, ip_)
    np.testing.assert_allclose([r0, p0, y0], [2.2, -0.7, 1.5], atol=1e-9)
    for order, euler in (("yaw,pitch,roll", "zxy"), ("pitch,roll,yaw", "xyz"), ("roll,yaw,pitch", "yzx")):
        t, y, p, r = mt.align_points(mp_, ip_, axes_order=order)
        expect = Rotation.from_matrix(R).as_euler(euler, degrees=True)
        np.testing.assert_allclose([r, p, y], expect, atol=1e-9, err_msg=order)
        np.testing.assert_allclose([t.x, t.y, t.z], [t0.x, t0.y, t0.z], atol=1e-12)
        # the three angles, applied in that extrinsic order, reproduce the rigid motion
        np.testing.assert_allclose(Rotation.from_euler(euler, [r, p, y], degrees=True).as_matrix(), R, atol=1e-12)
    with pytest.raises(KeyError):
        mt.align_points(mp_, ip_, axes_order="roll,pitch,spin")
    gold = np.load("tests/golden/fresh_golden.npz")
    for order in fc.ALIGN_ORDERS:
        t, y, p, r = mt.align_points(mp_, ip_, axes_order=order)
        np.testing.assert_allclose([y, p, r, t.x, t.y, t.z], gold[f"align_points/{order}"], atol=1e-9, err_msg=order)
