"""CPU: the PF oracle restatement against the reference's OWN fixtures -- the seven generated DICOM frames of
docs/source/files/ analysed with their docs recipes (docs/source/picketfence.rst:455-730).  Golden outputs come from the
UNMODIFIED reference (tests/golden/make_pf_docs_golden.py); the known answers printed in the docs (5 pickets / 250 kisses /
zero error for the perfect images, offsets 79.8 39.8 -0.2 -40.2 -80.1 mm) are asserted as well."""
import hashlib
import warnings

import numpy as np
import pytest

from oracle import pf_oracle
from tests.golden import pf_docs_cases as dc
from tests.test_oracle_pf import CLOSE, EXACT

GOLD = np.load("tests/golden/pf_docs_golden.npz")


@pytest.mark.parametrize("name", list(dc.DOCS))
def test_oracle_matches_reference_on_docs_fixture(name):
    a, ps, sid, ak = dc.docs_frame(name)
    sha = np.frombuffer(hashlib.sha1(a.tobytes()).digest(), dtype=np.uint8)
    assert np.array_equal(sha, GOLD[f"{name}/input_sha1"])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        o = pf_oracle.pf_analyze(a, (1 / ps) * sid / 1000.0, **ak)
    for k in EXACT:
        assert np.array_equal(np.asarray(o[k]), GOLD[f"{name}/{k}"]), k
    for k in CLOSE:
        np.testing.assert_array_equal(np.asarray(o[k]), GOLD[f"{name}/{k}"], err_msg=k)
    assert str(o["max_error_leaf"]) == str(GOLD[f"{name}/max_error_leaf"])
    assert [str(x) for x in o["failed_leaves"]] == [str(x) for x in GOLD[f"{name}/failed_leaves"]]


@pytest.mark.parametrize("name", ["perfect_up_down", "perfect_left_right"])
def test_docs_known_answers(name):
    """docs/source/picketfence.rst:497-505, 530-538: perfect images -> 5 pickets, 250 kisses, no error, 40 mm spacing."""
    g = lambda k: GOLD[f"{name}/{k}"]
    assert int(g("number_of_pickets")) == 5 and int(g("n_meas")) == 250 and bool(g("passed"))
    assert float(g("max_error")) < 1e-9
    np.testing.assert_allclose(g("offsets_from_cax_mm"), [79.8, 39.8, -0.2, -40.2, -80.1], atol=0.06)
    assert int(g("orientation")) == (0 if name == "perfect_up_down" else 1)
