"""CPU: the oracle restatements against the UNMODIFIED reference on fresh seeded frames that are not part of the per-module goldens
-- those pin fixed cases, this guards against an oracle that only fits them.  The reference's outputs for these frames are stored
in tests/golden/fresh_golden.npz (tests/golden/make_fresh_golden.py); each test first checks that it regenerated the same frame."""
import hashlib
import warnings

import numpy as np
import pytest

from tests.golden import fresh_cases as fc

GOLD = np.load("tests/golden/fresh_golden.npz")


def _same_input(group, seed, a):
    sha = np.frombuffer(hashlib.sha1(a.tobytes()).digest(), dtype=np.uint8)
    assert np.array_equal(sha, GOLD[f"{group}/{seed}/input_sha1"]), "the seeded frame differs from the one the reference analysed"


@pytest.mark.parametrize("seed", fc.PF_SEEDS)
def test_pf_oracle_equals_reference_on_fresh_frames(seed):
    from oracle import pf_oracle
    from tests.test_oracle_pf import CLOSE, EXACT

    a, ps = fc.pf_frame(seed)
    _same_input("pf", seed, a)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        o = pf_oracle.pf_analyze(a, 1 / ps)
    for k in EXACT:
        assert np.array_equal(np.asarray(o[k]), GOLD[f"pf/{seed}/{k}"]), k
    for k in CLOSE:
        np.testing.assert_array_equal(np.asarray(o[k]), GOLD[f"pf/{seed}/{k}"], err_msg=k)


@pytest.mark.parametrize("seed", fc.STAR_SEEDS)
def test_starshot_oracle_equals_reference_on_fresh_frames(seed):
    from oracle import starshot_oracle

    a, ps = fc.starshot_frame(seed)
    _same_input("star", seed, a)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        o = starshot_oracle.starshot_analyze(a, 1 / ps)
    for k in ("iterations", "profile_len", "peak_idx", "n_lines", "passed"):
        assert np.array_equal(np.asarray(o[k]), GOLD[f"star/{seed}/{k}"]), k
    for k in ("wobble_center", "wobble_radius_px", "angles"):
        np.testing.assert_allclose(np.asarray(o[k]), GOLD[f"star/{seed}/{k}"], rtol=1e-12, atol=1e-12, err_msg=k)


@pytest.mark.parametrize("seed", fc.FIELD_SEEDS)
def test_field_oracle_equals_reference_on_fresh_frames(seed):
    from oracle import field_oracle

    a, ps = fc.field_frame(seed)
    _same_input("field", seed, a)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        o = field_oracle.field_analyze(a, 1 / ps)
    for k in ("field_size_horizontal_mm", "field_size_vertical_mm", "beam_center_index_x_y", "left_penumbra_mm", "top_penumbra_mm",
              "flatness_horizontal", "symmetry_vertical", "cax_to_left_mm", "cax_to_top_mm"):
        np.testing.assert_allclose(np.asarray(o[k], dtype=float), GOLD[f"field/{seed}/{k}"], rtol=0, atol=1e-7, err_msg=k)


@pytest.mark.parametrize("seed", fc.WL_SEEDS)
def test_wl_oracle_equals_reference_on_fresh_frames(seed):
    from oracle import wl_oracle

    a, ps, _, _ = fc.wl_frame(seed)
    _same_input("wl", seed, a)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        o = wl_oracle.wl2d_analyze(a, 1 / ps)
    for k in ("field_cax", "bb", "epid", "cax2bb_vector", "cax2bb_distance", "cax2epid_distance"):
        np.testing.assert_allclose(np.asarray(o[k], dtype=float), GOLD[f"wl/{seed}/{k}"], rtol=0, atol=1e-9, err_msg=k)
