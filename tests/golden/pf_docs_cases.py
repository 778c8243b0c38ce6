"""The reference's own PicketFence fixtures: the seven generated DICOM files under docs/source/files/ with the analyze() calls of
their recipes (docs/source/picketfence.rst:455-730).  1280 x 1280, AS1200 pitch 0.336 mm, SID 1000.

All seven FILES (header + pixel data, lzma-compressed, ~10 MB together) are committed in tests/golden/pf_docs_dcm.npz; the GPU
tests run every fixture from there, and the file-level tests read them through pylinac_b200.dicom.
"""
from __future__ import annotations

import lzma
import os

import numpy as np

DCM_NPZ = os.path.join(os.path.dirname(__file__), "pf_docs_dcm.npz")
PIXEL_MM, SHAPE = 0.336, (1280, 1280)
# RTImageSID of each file (the docs recipes build three of them with AS1200Image(sid=1500), docs/source/picketfence.rst:551-667);
# tests/test_dicom_host.py checks these against the tags of the committed files
SID = {"perfect_up_down": 1000.0, "perfect_left_right": 1000.0, "noisy_wide_gap_up_down": 1500.0, "separated_wide_gap_up_down": 1500.0,
       "rotated_up_down": 1500.0, "offset_picket": 1000.0, "erroneous_leaves": 1000.0}

DOCS = {
    # name: analyze kwargs of the docs recipe
    "perfect_up_down": {"separate_leaves": False, "nominal_gap_mm": 4},
    "perfect_left_right": {"separate_leaves": False, "nominal_gap_mm": 4},
    "noisy_wide_gap_up_down": {},
    "separated_wide_gap_up_down": {"separate_leaves": True, "nominal_gap_mm": 10},
    "rotated_up_down": {"separate_leaves": False, "nominal_gap_mm": 5},
    "offset_picket": {},
    "erroneous_leaves": {"separate_leaves": True, "nominal_gap_mm": 5},
}


def _pixel_tail(data: bytes):
    """Uncompressed little-endian DICOM: PixelData is the last element (SURVEY.md section 0 fact 8)."""
    n = SHAPE[0] * SHAPE[1] * 2
    return np.frombuffer(data[-n:], dtype=np.uint16).reshape(SHAPE).copy()


def docs_dcm_bytes(name) -> bytes:
    """The complete DICOM file of a docs fixture."""
    with np.load(DCM_NPZ) as z:
        return lzma.decompress(z[name].tobytes())


def docs_frame(name):
    """-> (frame uint16 [1280,1280], pixel_spacing_mm, sid, analyze_kwargs)"""
    return _pixel_tail(docs_dcm_bytes(name)), PIXEL_MM, SID[name], dict(DOCS[name])
