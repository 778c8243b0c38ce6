"""Generate tests/golden/fresh_golden.npz by running the UNMODIFIED reference (stub-imported, oracle/refstub.py) on the seeded inputs
of fresh_cases.py: PicketFence, Starshot, FieldAnalysis and WinstonLutz2D on fresh frames, bb_projection_with_rotation on 300 random
setups and align_points in three axes orders.  Only the quantities the tests compare are stored.

Run where the reference tree is importable:  python -m tests.golden.make_fresh_golden
"""
from __future__ import annotations

import hashlib
import sys
import warnings

import numpy as np

from tests.golden import fresh_cases as fc
from tests.golden.refrun import reference_field, reference_pf, reference_starshot, reference_wl2d

PF_KEYS = ["orientation", "n_meas", "meas_leaf", "meas_picket", "picket_idx", "max_error_picket", "passed", "number_of_pickets",
           "meas_position", "meas_error", "meas_width_mm", "picket_spacing", "fits", "percent_passing", "max_error",
           "abs_median_error", "offsets_from_cax_mm", "mean_picket_spacing", "mlc_skew", "picket_widths"]
STAR_KEYS = ["iterations", "profile_len", "peak_idx", "n_lines", "passed", "wobble_center", "wobble_radius_px", "angles"]
FIELD_KEYS = ["field_size_horizontal_mm", "field_size_vertical_mm", "beam_center_index_x_y", "left_penumbra_mm", "top_penumbra_mm",
              "flatness_horizontal", "symmetry_vertical", "cax_to_left_mm", "cax_to_top_mm"]
WL_KEYS = ["field_cax", "bb", "epid", "cax2bb_vector", "cax2bb_distance", "cax2epid_distance"]


def _sha1(a):
    return np.frombuffer(hashlib.sha1(a.tobytes()).digest(), dtype=np.uint8)


def main():
    from oracle.refstub import import_reference

    warnings.simplefilter("ignore")
    store = {}
    for seed in fc.PF_SEEDS:
        a, ps = fc.pf_frame(seed)
        ref = reference_pf(a, ps, 1000.0, {}, {})
        store[f"pf/{seed}/input_sha1"] = _sha1(a)
        store.update({f"pf/{seed}/{k}": np.asarray(ref[k]) for k in PF_KEYS})
    for seed in fc.STAR_SEEDS:
        a, ps = fc.starshot_frame(seed)
        ref = reference_starshot(a, ps, 1000.0)
        store[f"star/{seed}/input_sha1"] = _sha1(a)
        store.update({f"star/{seed}/{k}": np.asarray(ref[k]) for k in STAR_KEYS})
    for seed in fc.FIELD_SEEDS:
        a, ps = fc.field_frame(seed)
        ref = reference_field(a, ps, 1000.0)
        store[f"field/{seed}/input_sha1"] = _sha1(a)
        store.update({f"field/{seed}/{k}": np.asarray(ref[k], dtype=float) for k in FIELD_KEYS})
    for seed in fc.WL_SEEDS:
        a, ps, g, p = fc.wl_frame(seed)
        ref = reference_wl2d(a, ps, 1000.0, g, 0.0, p)
        store[f"wl/{seed}/input_sha1"] = _sha1(a)
        store.update({f"wl/{seed}/{k}": np.asarray(ref[k], dtype=float) for k in WL_KEYS})

    import_reference()
    from pylinac import winston_lutz as rwl

    x = fc.bb_projection_inputs()
    store["bb_projection/inputs"] = x
    store["bb_projection/outputs"] = np.array([rwl.bb_projection_with_rotation(*row) for row in x], dtype=np.float64)
    pts, moved = fc.align_points_inputs()
    for order in fc.ALIGN_ORDERS:
        t, y, p, r = rwl.align_points([rwl.Point(*q) for q in pts], [rwl.Point(*q) for q in moved], axes_order=order)
        store[f"align_points/{order}"] = np.array([y, p, r, t.x, t.y, t.z], dtype=np.float64)
    np.savez_compressed("tests/golden/fresh_golden.npz", **store)
    print(len(store), "arrays")


if __name__ == "__main__":
    sys.exit(main())
