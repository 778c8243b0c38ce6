"""Contrast definitions -- mirror of ``pylinac.core.contrast`` (core/contrast.py:8-137).

Scalar host arithmetic on ROI results (pixel values, medians, standard deviations): the same formulas, the same numpy calls and the
same exceptions as the reference, so that a contrast computed from device statistics rounds exactly like the reference's."""
from __future__ import annotations

import numpy as np


class OptionListMixin:
    """The class attributes of an enum-like class as a list (core/utilities.py:35-45)."""

    @classmethod
    def options(cls) -> list[str]:
        return [option for attr, option in cls.__dict__.items() if not callable(option) and not attr.startswith("__")]


class Contrast(OptionListMixin):
    """Contrast calculation technique (core/contrast.py:8-15)."""

    MICHELSON = "Michelson"  #:
    WEBER = "Weber"  #:
    RATIO = "Ratio"  #:
    RMS = "Root Mean Square"  #:
    DIFFERENCE = "Difference"  #:


def visibility(array: np.ndarray, radius: float, std: float, algorithm: str) -> float:
    """The Rose-model visibility: contrast * sqrt(pi r^2) / std (core/contrast.py:18-40)."""
    c = contrast(array, algorithm)
    return c * np.sqrt(radius**2 * np.pi) / std


def contrast(array: np.ndarray, algorithm: str) -> float:
    """Dispatch on the (case-insensitive) algorithm name (core/contrast.py:43-84).  Weber, Ratio and Difference take a 2-element
    array (feature, background)."""
    algorithm = algorithm.lower()
    if algorithm == Contrast.MICHELSON.lower():
        return michelson(array)
    elif algorithm == Contrast.WEBER.lower():
        if array.size != 2:
            raise ValueError("For Weber algorithm, the array must be exactly 2 elements. Consult the ``weber`` function for parameter details")
        return weber(array[0], array[1])
    elif algorithm == Contrast.RMS.lower():
        return rms(array)
    elif algorithm == Contrast.RATIO.lower():
        if array.size != 2:
            raise ValueError("For Ratio algorithm, the array must be exactly 2 elements. Consult the ``ratio`` function for parameter details")
        return ratio(array[0], array[1])
    elif algorithm == Contrast.DIFFERENCE.lower():
        if array.size != 2:
            raise ValueError(
                "For Difference algorithm, the array must be exactly 2 elements. Consult the ``difference`` function for parameter details")
        return difference(array[0], array[1])
    else:
        raise ValueError(f"Contrast input of {algorithm} did not match any valid options: {Contrast.__dict__.values()}")


def rms(array: np.ndarray) -> float:
    """Root-mean-square contrast; the values must lie in [0, 1] (core/contrast.py:87-93)."""
    if array.min() < 0 or array.max() > 1:
        raise ValueError("RMS calculations require the input array to be normalized. I.e. only values between 0 and 1.")
    return np.sqrt(np.mean((array - array.mean()) ** 2))


def difference(feature: float, background: float) -> float:
    """|feature - background| (core/contrast.py:96-105)."""
    return abs(feature - background)


def michelson(array: np.ndarray) -> float:
    """(max - min) / (max + min), NaN-ignoring (core/contrast.py:108-116)."""
    l_max, l_min = np.nanmax(array), np.nanmin(array)
    return (l_max - l_min) / (l_max + l_min)


def weber(feature: float, background: float) -> float:
    """|feature - background| / background: the absolute difference, as the reference keeps it (core/contrast.py:119-132)."""
    return abs(feature - background) / background


def ratio(feature: float, reference: float) -> float:
    """feature / reference (core/contrast.py:135-137)."""
    return feature / reference
