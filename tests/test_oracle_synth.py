"""The restated image generator (oracle/synth.py, test infrastructure) against the pieces of the reference's generator that run
without scikit-image: the BB projection of generate_winstonlutz (winston_lutz.py:3401-3460), whose outputs on 300 random setups are
stored in tests/golden/fresh_golden.npz (tests/golden/make_fresh_golden.py)."""
import numpy as np

from oracle import synth
from tests.golden import fresh_cases as fc


def test_bb_projection_matches_the_reference_function():
    gold = np.load("tests/golden/fresh_golden.npz")
    x = gold["bb_projection/inputs"]
    np.testing.assert_array_equal(x, fc.bb_projection_inputs())
    ours = np.array([synth.bb_projection_with_rotation(*row) for row in x])
    assert np.max(np.abs(ours - gold["bb_projection/outputs"])) < 1e-12
