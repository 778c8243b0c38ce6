"""Seeded inputs that are not part of the per-module golden cases: the oracle restatements are checked on them against outputs of the
UNMODIFIED reference stored in fresh_golden.npz (make_fresh_golden.py), so an oracle that only fits the module cases shows up."""
from __future__ import annotations

import numpy as np

from oracle import synth

PF_SEEDS, STAR_SEEDS, FIELD_SEEDS, WL_SEEDS = (901, 902, 903), (911, 912), (921, 922), (931, 932)
ALIGN_ORDERS = ("roll,pitch,yaw", "yaw,pitch,roll", "pitch,roll,yaw")


def pf_frame(seed):
    """-> (frame uint16, pixel_spacing_mm)"""
    rng = np.random.default_rng(seed)
    fr = synth.epid1024()
    a = synth.picketfence_frame(fr, pickets=int(rng.integers(5, 11)), picket_spacing_mm=int(rng.integers(18, 28)),
                                picket_width_mm=int(rng.integers(2, 5)), picket_offset_error=rng.uniform(-0.6, 0.6, 12),
                                noise_sigma=float(rng.uniform(0.001, 0.004)), seed=seed,
                                orientation="left_right" if seed % 2 else "up_down")
    return a, fr.pixel_size


def starshot_frame(seed):
    """-> (frame uint16, pixel_spacing_mm)"""
    rng = np.random.default_rng(seed)
    spokes = int(rng.choice([4, 6, 8]))
    fr = synth.epid1024()
    a = synth.starshot_frame(fr, spokes=spokes, offsets_mm=[tuple(rng.uniform(-0.6, 0.6, 2)) for _ in range(spokes)],
                             noise_sigma=0.003, seed=seed)
    return a, fr.pixel_size


def field_frame(seed):
    """-> (frame uint16, pixel_spacing_mm)"""
    rng = np.random.default_rng(seed)
    fr = synth.as1200(1000.0)
    a = synth.openfield_frame(fr, field_size_mm=(int(rng.integers(80, 200)), int(rng.integers(80, 200))),
                              cax_offset_mm=tuple(rng.uniform(-8, 8, 2)), seed=seed)
    return a, fr.pixel_size


def wl_frame(seed):
    """-> (frame uint16, pixel_spacing_mm, gantry, couch)"""
    rng = np.random.default_rng(seed)
    fr = synth.epid1024()
    g, p = float(rng.integers(0, 360)), float(rng.choice([0, 45, 315]))
    a = synth.winstonlutz_frame(fr, offset_mm_left=rng.uniform(-1.5, 1.5), offset_mm_up=rng.uniform(-1.5, 1.5),
                                offset_mm_in=rng.uniform(-1.5, 1.5), gantry=g, couch=p, noise_sigma=0.003, seed=seed)
    return a, fr.pixel_size, g, p


def bb_projection_inputs():
    """[300, 5]: (left, up, in) mm in [-5, 5], gantry and couch degrees in [0, 360)."""
    rng = np.random.default_rng(0)
    return np.array([np.concatenate([rng.uniform(-5, 5, 3), rng.uniform(0, 360, 2)]) for _ in range(300)])


def align_points_inputs():
    """-> (points [7, 3], the same points after a rigid motion)"""
    from scipy.spatial.transform import Rotation

    rng = np.random.default_rng(9)
    pts = rng.uniform(-50, 50, size=(7, 3))
    R = Rotation.from_euler("yxz", [2.2, -0.7, 1.5], degrees=True).as_matrix()
    return pts, pts @ R.T + np.array([0.4, -1.1, 2.0])
