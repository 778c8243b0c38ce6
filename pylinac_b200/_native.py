"""ctypes binding of ``libepid.so`` (the C-ABI declared in ``include/epid.h``).

This is the only module that touches the native library.  There is NO CPU fallback: if the shared
library is missing, or no CUDA device is visible, the compute entry points raise.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EPID_LIB") or os.path.join(_HERE, "libepid.so")      # EPID_LIB: kernel-variant experiments (tools/)

EPID_OK = 0
ERR_NO_DEVICE, ERR_CUDA, ERR_INVALID, ERR_UNSUPPORTED, ERR_NOMEM, ERR_NCCL, ERR_INDEX = -1, -2, -3, -4, -5, -6, -7

U8, U16, I32, F32, F64, I16, I64 = 0, 1, 2, 3, 4, 5, 6
_NP2DT = {np.dtype(np.uint8): U8, np.dtype(np.uint16): U16, np.dtype(np.int32): I32, np.dtype(np.float32): F32,
          np.dtype(np.float64): F64, np.dtype(np.int16): I16, np.dtype(np.int64): I64}
_DT2NP = {v: k for k, v in _NP2DT.items()}

OPT_PF_EXACT_ONLY = 1
OPT_PF_WIN2 = 3
OPT_PF_FAST_REDO = 5
OPT_STATS_EXACT = 7
CTR_PF_FALLBACKS = 1
CTR_PF_REDONE_FRAMES = 2
CTR_PF_EXACT_FRAMES = 3
CTR_STATS_UNCERTIFIED = 4
PF_MAX_PICKETS = 32
PF_MAX_LEAVES = 160


class NativeError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libepid error {code}: {msg}")
        self.code = code
        self.msg = msg


class NoDeviceError(NativeError):
    pass


class PeakParams(C.Structure):
    _fields_ = [("threshold", C.c_double), ("peak_separation", C.c_double), ("max_number", C.c_int32),
                ("fwxm_height", C.c_double), ("min_width", C.c_double), ("search_lo", C.c_double),
                ("search_hi", C.c_double), ("peak_sort", C.c_int32), ("required_prominence", C.c_double)]


class PFParams(C.Structure):
    _fields_ = [("dpmm", C.c_double), ("crop_px", C.c_int32), ("filter_size", C.c_int32), ("tolerance", C.c_double),
                ("action_tolerance", C.c_double), ("num_pickets", C.c_int32), ("sag_px", C.c_int32),
                ("orientation", C.c_int32), ("invert", C.c_int32), ("leaf_analysis_width_ratio", C.c_double),
                ("picket_spacing", C.c_double), ("height_threshold", C.c_double), ("edge_threshold", C.c_double),
                ("peak_sort", C.c_int32), ("required_prominence", C.c_double), ("separate_leaves", C.c_int32),
                ("nominal_gap_mm", C.c_double), ("has_cax_override", C.c_int32), ("cax_x_px", C.c_double),
                ("cax_y_px", C.c_double), ("n_leaves", C.c_int32), ("leaf_center_mm", C.c_double * PF_MAX_LEAVES),
                ("leaf_width_mm", C.c_double * PF_MAX_LEAVES), ("leaf_num", C.c_int32 * PF_MAX_LEAVES)]


class PFSummary(C.Structure):
    _fields_ = [("status", C.c_int32), ("orientation", C.c_int32), ("noise_median_passes", C.c_int32),
                ("corner_inverted", C.c_int32), ("height", C.c_int32), ("width", C.c_int32), ("n_pickets", C.c_int32),
                ("n_meas", C.c_int32), ("n_leaves_removed", C.c_int32), ("passed", C.c_int32),
                ("max_error_picket", C.c_int32), ("max_error_leaf", C.c_int32), ("max_error_bank", C.c_int32),
                ("n_failed", C.c_int32), ("picket_spacing_px", C.c_double), ("percent_passing", C.c_double),
                ("max_error_mm", C.c_double), ("abs_median_error_mm", C.c_double), ("mean_picket_spacing_mm", C.c_double),
                ("mlc_skew", C.c_double), ("cax_px", C.c_double), ("picket_idx", C.c_int32 * PF_MAX_PICKETS),
                ("picket_val", C.c_double * PF_MAX_PICKETS), ("fit_slope", C.c_double * PF_MAX_PICKETS),
                ("fit_intercept", C.c_double * PF_MAX_PICKETS), ("offsets_from_cax_mm", C.c_double * PF_MAX_PICKETS),
                ("picket_width_max", C.c_double * PF_MAX_PICKETS), ("picket_width_mean", C.c_double * PF_MAX_PICKETS),
                ("picket_width_median", C.c_double * PF_MAX_PICKETS), ("picket_width_min", C.c_double * PF_MAX_PICKETS)]


class PFMeas(C.Structure):
    _fields_ = [("leaf_num", C.c_int32), ("picket", C.c_int32), ("passed", C.c_int32 * 2), ("position", C.c_double * 2),
                ("error", C.c_double * 2), ("width_mm", C.c_double)]


PF_SUMMARY_DTYPE = np.dtype([
    ("status", "<i4"), ("orientation", "<i4"), ("noise_median_passes", "<i4"), ("corner_inverted", "<i4"),
    ("height", "<i4"), ("width", "<i4"), ("n_pickets", "<i4"), ("n_meas", "<i4"), ("n_leaves_removed", "<i4"),
    ("passed", "<i4"), ("max_error_picket", "<i4"), ("max_error_leaf", "<i4"), ("max_error_bank", "<i4"),
    ("n_failed", "<i4"), ("picket_spacing_px", "<f8"), ("percent_passing", "<f8"), ("max_error_mm", "<f8"),
    ("abs_median_error_mm", "<f8"), ("mean_picket_spacing_mm", "<f8"), ("mlc_skew", "<f8"), ("cax_px", "<f8"),
    ("picket_idx", "<i4", (PF_MAX_PICKETS,)), ("picket_val", "<f8", (PF_MAX_PICKETS,)),
    ("fit_slope", "<f8", (PF_MAX_PICKETS,)), ("fit_intercept", "<f8", (PF_MAX_PICKETS,)),
    ("offsets_from_cax_mm", "<f8", (PF_MAX_PICKETS,)), ("picket_width_max", "<f8", (PF_MAX_PICKETS,)),
    ("picket_width_mean", "<f8", (PF_MAX_PICKETS,)), ("picket_width_median", "<f8", (PF_MAX_PICKETS,)),
    ("picket_width_min", "<f8", (PF_MAX_PICKETS,))], align=True)
PF_MEAS_DTYPE = np.dtype([("leaf_num", "<i4"), ("picket", "<i4"), ("passed", "<i4", (2,)), ("position", "<f8", (2,)),
                          ("error", "<f8", (2,)), ("width_mm", "<f8")], align=True)
assert PF_SUMMARY_DTYPE.itemsize == C.sizeof(PFSummary), (PF_SUMMARY_DTYPE.itemsize, C.sizeof(PFSummary))
assert PF_MEAS_DTYPE.itemsize == C.sizeof(PFMeas)

STAR_MAX_PEAKS = 64


class StarParams(C.Structure):
    _fields_ = [("dpmm", C.c_double), ("radius", C.c_double), ("min_peak_height", C.c_double), ("max_wobble_diameter", C.c_double),
                ("tolerance", C.c_double), ("has_start_point", C.c_int32), ("start_x", C.c_double), ("start_y", C.c_double),
                ("fwhm", C.c_int32), ("recursive", C.c_int32), ("invert", C.c_int32)]


class StarResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("hist_inverted", C.c_int32), ("start_x", C.c_int32), ("start_y", C.c_int32),
                ("local_max", C.c_double), ("iterations", C.c_int32), ("profile_len", C.c_int32), ("radius_px", C.c_double),
                ("n_peaks", C.c_int32), ("n_lines", C.c_int32), ("peak_idx", C.c_int32 * STAR_MAX_PEAKS),
                ("peak_x", C.c_double * STAR_MAX_PEAKS), ("peak_y", C.c_double * STAR_MAX_PEAKS), ("wobble_x", C.c_double),
                ("wobble_y", C.c_double), ("wobble_radius_px", C.c_double), ("wobble_radius_mm", C.c_double),
                ("angles", C.c_double * (STAR_MAX_PEAKS // 2)), ("passed", C.c_int32), ("pad", C.c_int32)]


STAR_RESULT_DTYPE = np.dtype([
    ("status", "<i4"), ("hist_inverted", "<i4"), ("start_x", "<i4"), ("start_y", "<i4"), ("local_max", "<f8"),
    ("iterations", "<i4"), ("profile_len", "<i4"), ("radius_px", "<f8"), ("n_peaks", "<i4"), ("n_lines", "<i4"),
    ("peak_idx", "<i4", (STAR_MAX_PEAKS,)), ("peak_x", "<f8", (STAR_MAX_PEAKS,)), ("peak_y", "<f8", (STAR_MAX_PEAKS,)),
    ("wobble_x", "<f8"), ("wobble_y", "<f8"), ("wobble_radius_px", "<f8"), ("wobble_radius_mm", "<f8"),
    ("angles", "<f8", (STAR_MAX_PEAKS // 2,)), ("passed", "<i4"), ("pad", "<i4")], align=True)
assert STAR_RESULT_DTYPE.itemsize == C.sizeof(StarResult), (STAR_RESULT_DTYPE.itemsize, C.sizeof(StarResult))

class FieldParams(C.Structure):
    _fields_ = [("dpmm", C.c_double), ("protocol", C.c_int32), ("centering", C.c_int32), ("vert_position", C.c_double),
                ("horiz_position", C.c_double), ("vert_width", C.c_double), ("horiz_width", C.c_double),
                ("in_field_ratio", C.c_double), ("slope_exclusion_ratio", C.c_double), ("invert", C.c_int32),
                ("penumbra_lower", C.c_double), ("penumbra_upper", C.c_double), ("interpolation", C.c_int32),
                ("interpolation_resolution_mm", C.c_double), ("ground", C.c_int32), ("normalization", C.c_int32),
                ("edge", C.c_int32), ("edge_smoothing_ratio", C.c_double)]


_FIELD_DOUBLES = ["top_penumbra_mm", "bottom_penumbra_mm", "left_penumbra_mm", "right_penumbra_mm"]
_FIELD_LAYOUT = [
    ("status", "<i4"), ("hist_inverted", "<i4"), ("strip_rows", "<i4", (2,)), ("strip_cols", "<i4", (2,)), ("profile_len", "<i4", (2,)),
    ("top_penumbra_mm", "<f8"), ("bottom_penumbra_mm", "<f8"), ("left_penumbra_mm", "<f8"), ("right_penumbra_mm", "<f8"),
    ("geometric_center_index_x_y", "<f8", (2,)), ("beam_center_index_x_y", "<f8", (2,)),
    ("field_size_vertical_mm", "<f8"), ("field_size_horizontal_mm", "<f8"),
    ("beam_center_to_top_mm", "<f8"), ("beam_center_to_bottom_mm", "<f8"), ("beam_center_to_left_mm", "<f8"),
    ("beam_center_to_right_mm", "<f8"), ("cax_to_top_mm", "<f8"), ("cax_to_bottom_mm", "<f8"), ("cax_to_left_mm", "<f8"),
    ("cax_to_right_mm", "<f8"), ("top_position_index_x_y", "<f8", (2,)),
    ("top_horizontal_distance_from_cax_mm", "<f8"), ("top_vertical_distance_from_cax_mm", "<f8"),
    ("top_horizontal_distance_from_beam_center_mm", "<f8"), ("top_vertical_distance_from_beam_center_mm", "<f8"),
    ("left_slope_percent_mm", "<f8"), ("right_slope_percent_mm", "<f8"), ("top_slope_percent_mm", "<f8"),
    ("bottom_slope_percent_mm", "<f8"), ("symmetry_horizontal", "<f8"), ("symmetry_vertical", "<f8"),
    ("flatness_horizontal", "<f8"), ("flatness_vertical", "<f8")]
FIELD_RESULT_DTYPE = np.dtype(_FIELD_LAYOUT, align=True)


def _struct_from_layout(name, layout):
    fields = []
    for item in layout:
        ct = C.c_int32 if item[1] == "<i4" else C.c_double
        fields.append((item[0], ct * item[2][0] if len(item) == 3 else ct))
    return type(name, (C.Structure,), {"_fields_": fields})


FieldResult = _struct_from_layout("FieldResult", _FIELD_LAYOUT)
assert FIELD_RESULT_DTYPE.itemsize == C.sizeof(FieldResult), (FIELD_RESULT_DTYPE.itemsize, C.sizeof(FieldResult))

class SpParams(C.Structure):
    _fields_ = [("dpmm", C.c_double), ("interpolation", C.c_int32), ("interpolation_resolution_mm", C.c_double),
                ("interpolation_factor", C.c_double), ("ground", C.c_int32), ("normalization", C.c_int32), ("edge", C.c_int32),
                ("centering", C.c_int32), ("edge_smoothing_ratio", C.c_double), ("x_start", C.c_double), ("x_stop", C.c_double),
                ("edge_left", C.c_double), ("edge_right", C.c_double)]


_SP_LAYOUT = [
    ("status", "<i4"), ("n", "<i4"), ("x_start", "<f8"), ("x_stop", "<f8"), ("values_max", "<f8"),
    ("geometric_center_index", "<f8"), ("geometric_center_value", "<f8"),
    ("beam_ok", "<i4"), ("fwxm_ok", "<i4"), ("infl_ok", "<i4"), ("pen_ok", "<i4"), ("fd_ok", "<i4"), ("fd_field_values_n", "<i4"),
    ("beam_center_index", "<f8"), ("beam_center_value_at_rounded", "<f8"),
    ("fwxm_left", "<f8"), ("fwxm_right", "<f8"), ("fwxm_center_value_at_rounded", "<f8"), ("fwxm_left_value_at_rounded", "<f8"),
    ("fwxm_right_value_at_rounded", "<f8"),
    ("infl_left", "<f8"), ("infl_right", "<f8"), ("infl_left_value_exact", "<f8"), ("infl_right_value_exact", "<f8"),
    ("infl_left_value_rounded", "<f8"), ("infl_right_value_rounded", "<f8"),
    ("pen_left_lower", "<f8"), ("pen_left_upper", "<f8"), ("pen_right_lower", "<f8"), ("pen_right_upper", "<f8"),
    ("fd_width", "<f8"), ("fd_beam_center", "<f8"), ("fd_cax", "<f8"), ("fd_left", "<f8"), ("fd_right", "<f8"),
    ("fd_inner_left", "<f8"), ("fd_inner_right", "<f8"), ("fd_left_slope", "<f8"), ("fd_left_intercept", "<f8"),
    ("fd_right_slope", "<f8"), ("fd_right_intercept", "<f8"), ("fd_top_index", "<f8"), ("fd_top_value", "<f8"),
    ("fd_top_params", "<f8", (3,)), ("fd_beam_center_value", "<f8"), ("fd_cax_value", "<f8"), ("fd_left_value", "<f8"),
    ("fd_right_value", "<f8")]
SP_RESULT_DTYPE = np.dtype(_SP_LAYOUT, align=True)


class WlParams(C.Structure):
    _fields_ = [("dpmm", C.c_double), ("bb_size_mm", C.c_double), ("low_density_bb", C.c_int32), ("open_field", C.c_int32),
                ("bb_proximity_mm", C.c_double)]


(WL_OK, WL_NO_BB, WL_MISMATCH, WL_NO_FIELD, WL_CAPACITY, WL_FLAT_IMAGE) = range(6)
_WL_LAYOUT = [
    ("status", "<i4"), ("inverted", "<i4"), ("crop_px", "<i4"), ("height", "<i4"), ("width", "<i4"), ("n_bbs", "<i4"),
    ("threshold_passes", "<i4"), ("pad", "<i4"), ("bb_x", "<f8"), ("bb_y", "<f8"), ("field_x", "<f8"), ("field_y", "<f8"),
    ("epid_x", "<f8"), ("epid_y", "<f8"), ("cax2bb_x", "<f8"), ("cax2bb_y", "<f8"), ("cax2bb_distance", "<f8"),
    ("cax2epid_x", "<f8"), ("cax2epid_y", "<f8"), ("cax2epid_distance", "<f8")]
WL_RESULT_DTYPE = np.dtype(_WL_LAYOUT, align=True)
assert WL_RESULT_DTYPE.itemsize == 128
DISK_MAX = 8


class DiskParams(C.Structure):
    """epid_disk_params (include/epid.h)"""

    _fields_ = [("dpmm", C.c_double), ("expected_x", C.c_double), ("expected_y", C.c_double), ("window_w", C.c_double),
                ("window_h", C.c_double), ("radius_mm", C.c_double), ("tolerance_mm", C.c_double), ("min_separation_px", C.c_double),
                ("invert", C.c_int32), ("max_number", C.c_int32), ("conditions", C.c_int32), ("pad", C.c_int32)]


DISK_RESULT_DTYPE = np.dtype([("status", np.int32), ("n_points", np.int32), ("n_regions", np.int32), ("passes", np.int32),
                              ("left", np.int32), ("top", np.int32), ("x", np.float64, DISK_MAX), ("y", np.float64, DISK_MAX),
                              ("r_area", np.float64, DISK_MAX), ("r_filled_area", np.float64, DISK_MAX),
                              ("r_perimeter", np.float64, DISK_MAX), ("r_convex_area", np.float64, DISK_MAX),
                              ("r_centroid_y", np.float64, DISK_MAX), ("r_centroid_x", np.float64, DISK_MAX),
                              ("r_wcentroid_y", np.float64, DISK_MAX), ("r_wcentroid_x", np.float64, DISK_MAX),
                              ("r_bbox", np.int32, (DISK_MAX, 4))], align=True)
assert DISK_RESULT_DTYPE.itemsize == 24 + 8 * DISK_MAX * 10 + 4 * DISK_MAX * 4
_lib = None
_lock = threading.Lock()


def build(force: bool = False) -> str:
    """Compile libepid.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    src = os.path.join(_HERE, "csrc")
    if force:
        subprocess.run(["make", "-C", src, "clean"], check=True, stdout=subprocess.DEVNULL)
    subprocess.run(["make", "-C", src, "-j8"], check=True, stdout=subprocess.DEVNULL)
    return LIB_PATH


VMAT_MAX_SEG = 16


class VmatParams(C.Structure):
    _fields_ = [("ground", C.c_int32), ("check_inversion", C.c_int32), ("invert_image_order", C.c_int32), ("nseg", C.c_int32),
                ("dpmm", C.c_double), ("tolerance_percent", C.c_double), ("seg_w_mm", C.c_double), ("seg_h_mm", C.c_double),
                ("offset_mm", C.c_double * VMAT_MAX_SEG)]


_S = (VMAT_MAX_SEG,)
VMAT_RESULT_DTYPE = np.dtype([
    ("status", "<i4"), ("open_is_first", "<i4"), ("inverted", "<i4", (2,)), ("center_warning", "<i4"), ("passed", "<i4"), ("nseg", "<i4"),
    ("pad_", "<i4"), ("x_field_center", "<f8"), ("profile_center_idx", "<f8", (2,)), ("field_len", "<f8", (2,)), ("field_std", "<f8", (2,)),
    ("r_corr", "<f8", _S), ("r_dev", "<f8", _S), ("stdev", "<f8", _S), ("center_x", "<f8", _S), ("center_y", "<f8", _S), ("npix", "<f8", _S),
    ("seg_passed", "<i4", _S), ("max_r_deviation", "<f8"), ("avg_abs_r_deviation", "<f8"), ("avg_r_deviation", "<f8")], align=True)



class LocateParams(C.Structure):
    _fields_ = [("mode", C.c_int32), ("invert", C.c_int32), ("sample_kind", C.c_int32), ("conditions", C.c_int32), ("dpmm", C.c_double),
                ("radius_mm", C.c_double), ("tolerance_mm", C.c_double), ("field_width_mm", C.c_double), ("field_height_mm", C.c_double),
                ("field_tolerance_mm", C.c_double), ("bb_size_mm", C.c_double), ("rad_size_mm", C.c_double)]


REGION_DTYPE = np.dtype([("threshold_index", "<i4"), ("label_root", "<i4"), ("bbox", "<i4", (4,)), ("area", "<f8"), ("area_filled", "<f8"),
                         ("perimeter", "<f8"), ("equivalent_diameter", "<f8"), ("centroid_y", "<f8"), ("centroid_x", "<f8"),
                         ("wcentroid_y", "<f8"), ("wcentroid_x", "<f8")], align=True)

_P = C.c_void_p
_SIGNATURES = {
    "epid_device_count": [C.POINTER(C.c_int32)],
    "epid_ctx_create": [C.c_int32, C.POINTER(_P)],
    "epid_ctx_destroy": [_P],
    "epid_sync": [_P],
    "epid_device_info": [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_size_t)],
    "epid_device_pci_bus_id": [C.c_int32, C.c_char_p, C.c_int32],
    "epid_launch_count": [_P, C.POINTER(C.c_int64)],
    "epid_version": [],
    "epid_set_option": [_P, C.c_int32, C.c_int64],
    "epid_get_counter": [_P, C.c_int32, C.POINTER(C.c_int64)],
    "epid_host_alloc": [C.c_size_t, C.POINTER(_P)],
    "epid_host_free": [_P],
    "epid_batch_upload": [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_P)],
    "epid_batch_alloc": [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_P)],
    "epid_batch_download": [_P, _P],
    "epid_batch_write": [_P, _P],
    "epid_batch_free": [_P],
    "epid_batch_shape": [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)],
    "epid_batch_device_ptr": [_P, C.POINTER(_P)],
    "epid_frame_stats": [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, C.c_int32, _P, _P, _P, _P, _P, _P],
    "epid_frame_histogram": [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P],
    "epid_invert": [_P, _P, C.POINTER(_P)],
    "epid_bit_invert": [_P, _P, C.POINTER(_P)],
    "epid_ground": [_P, _P, C.c_double, C.POINTER(_P), _P],
    "epid_normalize": [_P, _P, C.c_int32, C.c_double, C.POINTER(_P)],
    "epid_threshold": [_P, _P, C.c_double, C.c_int32, C.POINTER(_P)],
    "epid_binarize": [_P, _P, C.c_double, C.POINTER(_P)],
    "epid_median_filter": [_P, _P, C.c_int32, C.POINTER(_P)],
    "epid_gaussian_filter": [_P, _P, C.c_double, C.POINTER(_P)],
    "epid_correlate1d_passes": [_P, _P, _P, C.c_int32, C.c_int32, C.POINTER(_P)],
    "epid_sobel": [_P, _P, C.c_int32, C.POINTER(_P)],
    "epid_find_peaks": [_P, _P, C.c_int32, C.POINTER(PeakParams), C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                        C.POINTER(C.c_int32)],
    "epid_pf_analyze": [_P, _P, C.POINTER(PFParams), _P, _P, C.c_int32],
    "epid_pf_analyze_host": [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(PFParams), _P, _P, C.c_int32],
    "epid_pf_bench": [_P, _P, C.POINTER(PFParams), C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float),
                      C.POINTER(C.c_int64)],
    "epid_pf_bench_timed": [_P, _P, C.POINTER(PFParams), C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_int32,
                            C.POINTER(C.c_int64), C.POINTER(C.c_int64)],
    "epid_starshot_analyze": [_P, _P, C.POINTER(StarParams), _P, _P, C.c_int32, _P],
    "epid_circle_profile": [_P, _P, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int32, C.c_double, C.c_int32, C.c_double,
                            C.c_int32, C.c_int32, _P, _P, _P, C.POINTER(C.c_int32)],
    "epid_single_profile": [_P, _P, _P, C.c_int32, C.POINTER(SpParams), _P, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_double,
                            C.c_double, C.c_double, _P, _P, _P, C.c_int32],
    "epid_field_profile_len": [C.c_int32, C.c_double, C.c_int32, C.c_double],
    "epid_field_analyze": [_P, _P, C.POINTER(FieldParams), _P, C.c_int32, _P, C.c_int32, _P],
    "epid_wl2d_analyze": [_P, _P, C.POINTER(WlParams), _P],
    "epid_zoom": [_P, _P, C.c_double, C.c_int32, C.c_int32, C.POINTER(_P)],
    "epid_rotate": [_P, _P, C.c_double, C.c_int32, C.POINTER(_P)],
    "epid_gamma": [_P, _P, _P, C.c_double, C.c_double, C.c_double, C.POINTER(_P)],
    "epid_disk_locate": [_P, _P, _P, _P],
    "epid_roi_stats": [_P, _P, C.c_int32, _P, _P, _P, _P, _P, _P],
    "epid_disk_roi_stats": [_P, _P, C.c_int32, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P],
    "epid_disk_roi_pixels": [_P, _P, C.c_int32, _P, C.c_double, C.c_int32, C.c_int64, _P, _P, _P, C.POINTER(C.c_int64)],
    "epid_weighted_centroid": [_P, _P, _P, _P, _P],
    "epid_vmat_analyze": [_P, _P, _P, C.POINTER(VmatParams), _P],
    "epid_divide": [_P, _P, _P, _P, C.POINTER(_P)],
    "epid_dlg_analyze": [_P, _P, C.c_int32, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P],
    "epid_global_locate": [_P, _P, C.POINTER(LocateParams), _P, C.c_int32, _P, _P],
    "epid_canny": [_P, _P, _P, C.c_int32, C.c_double, C.c_double, C.POINTER(_P)],
    "epid_hough_line": [_P, _P, C.c_int32, _P, C.POINTER(_P), C.POINTER(C.c_int32)],
    "epid_hough_candidates": [_P, _P, C.c_int32, C.c_int32, C.c_double, C.c_int32, _P, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                              C.POINTER(_P)],
    "epid_gather_i32": [_P, _P, C.c_int32, _P, _P],
    "epid_comm_unique_id": [_P],
    "epid_comm_init": [_P, C.c_int32, C.c_int32, _P],
    "epid_comm_destroy": [_P],
    "epid_comm_info": [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32)],
    "epid_gather_results": [_P, _P, C.c_size_t, _P],
    "epid_barrier": [_P],
}


def lib():
    """Load libepid.so (once).  Raises if the native extension has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise ImportError(
                        f"{LIB_PATH} is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(pylinac_b200 has no CPU fallback).")
                handle = C.CDLL(LIB_PATH)
                for name, args in _SIGNATURES.items():
                    fn = getattr(handle, name)
                    fn.argtypes = args
                    fn.restype = C.c_int32
                handle.epid_last_error.argtypes = []
                handle.epid_last_error.restype = C.c_char_p
                _lib = handle
    return _lib


def exported_symbols():
    return sorted(list(_SIGNATURES) + ["epid_last_error"])


def check(rc):
    if rc != EPID_OK:
        msg = lib().epid_last_error().decode("utf-8", "replace")
        if rc == ERR_NO_DEVICE:
            raise NoDeviceError(rc, msg)
        if rc == ERR_INVALID:
            raise ValueError(msg)
        if rc == ERR_INDEX:
            raise IndexError(msg)
        raise NativeError(rc, msg)


def device_count() -> int:
    n = C.c_int32(0)
    check(lib().epid_device_count(C.byref(n)))
    return n.value


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Context:
    """One per device (epid_ctx)."""

    _default = {}

    def __init__(self, device: int = 0):
        h = _P()
        check(lib().epid_ctx_create(device, C.byref(h)))
        self.handle = h
        self.device = device

    @classmethod
    def default(cls, device: int | None = None) -> "Context":
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0")) if device_count() > 1 else 0
            if device >= device_count():
                device = 0
        if device not in cls._default:
            cls._default[device] = cls(device)
        return cls._default[device]

    def close(self):
        if self.handle:
            lib().epid_ctx_destroy(self.handle)
            self.handle = None

    def sync(self):
        check(lib().epid_sync(self.handle))

    def info(self):
        sm, ma, mi, mem = C.c_int32(), C.c_int32(), C.c_int32(), C.c_size_t()
        check(lib().epid_device_info(self.handle, C.byref(sm), C.byref(ma), C.byref(mi), C.byref(mem)))
        return {"sm_count": sm.value, "cc": (ma.value, mi.value), "hbm_bytes": mem.value}

    def set_option(self, key: int, value: int) -> None:
        check(lib().epid_set_option(self.handle, key, value))

    def counter(self, key: int) -> int:
        v = C.c_int64()
        check(lib().epid_get_counter(self.handle, key, C.byref(v)))
        return v.value

    def comm_info(self) -> tuple[int, int]:
        """(nranks, rank) of this context's NCCL communicator; (1, 0) before parallel.init_comm."""
        n, r = C.c_int32(), C.c_int32()
        check(lib().epid_comm_info(self.handle, C.byref(n), C.byref(r)))
        return n.value, r.value

    def launches(self) -> int:
        n = C.c_int64()
        check(lib().epid_launch_count(self.handle, C.byref(n)))
        return n.value


class Batch:
    """n frames resident in HBM (epid_batch)."""

    def __init__(self, ctx: Context, handle):
        self.ctx = ctx
        self.handle = handle

    @classmethod
    def upload(cls, ctx: Context, arr: np.ndarray) -> "Batch":
        a = np.ascontiguousarray(arr)
        if a.ndim == 2:
            a = a[None]
        if a.ndim != 3:
            raise ValueError("expected [n, h, w] or [h, w]")
        if a.dtype not in _NP2DT:
            raise TypeError(f"unsupported dtype {a.dtype}")
        h = _P()
        check(lib().epid_batch_upload(ctx.handle, _ptr(a), _NP2DT[a.dtype], a.shape[0], a.shape[1], a.shape[2], C.byref(h)))
        return cls(ctx, h)

    @property
    def shape_dtype(self):
        dt, n, h, w = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        check(lib().epid_batch_shape(self.handle, C.byref(dt), C.byref(n), C.byref(h), C.byref(w)))
        return (n.value, h.value, w.value), _DT2NP[dt.value]

    def write(self, arr: np.ndarray) -> None:
        """overwrite the batch from a host array of the same shape / dtype (one H2D copy, synchronous)"""
        shape, dt = self.shape_dtype
        a = np.ascontiguousarray(arr)
        if a.shape != shape or a.dtype != dt:
            raise ValueError(f"expected {shape} {dt}, got {a.shape} {a.dtype}")
        check(lib().epid_batch_write(self.handle, _ptr(a)))

    def download(self) -> np.ndarray:
        shape, dt = self.shape_dtype
        out = np.empty(shape, dt)
        check(lib().epid_batch_download(self.handle, _ptr(out)))
        return out

    def free(self):
        if self.handle:
            lib().epid_batch_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def _unary2(self, fn, other: "Batch", *args) -> "Batch":
        h = _P()
        check(fn(self.ctx.handle, self.handle, other.handle, *args, C.byref(h)))
        return Batch(self.ctx, h)

    def _unary(self, fn, *args) -> "Batch":
        h = _P()
        check(fn(self.ctx.handle, self.handle, *args, C.byref(h)))
        return Batch(self.ctx, h)


def pinned_empty(shape, dtype=np.uint16) -> np.ndarray:
    """numpy array backed by page-locked host memory (epid_host_alloc); freed when the array dies."""
    dtype = np.dtype(dtype)
    nbytes = int(np.prod(shape)) * dtype.itemsize
    p = _P()
    check(lib().epid_host_alloc(nbytes, C.byref(p)))
    import weakref

    buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
    # every numpy view keeps `buf` alive through its .base chain; when the last one dies the block is unpinned and freed
    weakref.finalize(buf, _host_free, p.value)
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


def _host_free(ptr: int) -> None:
    try:
        lib().epid_host_free(_P(ptr))
    except Exception:
        pass


class _PinnedPool:
    """Page-locked result buffers, recycled between calls.  cudaHostAlloc costs milliseconds and a fresh pageable
    ``np.zeros`` of a 30 MB result block costs thousands of first-touch page faults per call; a pooled pinned block costs
    neither and lets the library DMA the results straight into the array the caller receives.  A block returns to the pool
    when the last numpy view of it is garbage collected."""

    MAX_FREE_PER_SIZE = 4

    def __init__(self):
        self._free: dict[int, list[int]] = {}
        self._lock = threading.Lock()

    def take(self, shape, dtype) -> np.ndarray:
        import weakref

        dtype = np.dtype(dtype)
        nbytes = max(int(np.prod(shape)) * dtype.itemsize, 1)
        with self._lock:
            lst = self._free.get(nbytes)
            ptr = lst.pop() if lst else None
        if ptr is None:
            p = _P()
            check(lib().epid_host_alloc(nbytes, C.byref(p)))
            ptr = p.value
        buf = (C.c_char * nbytes).from_address(ptr)
        weakref.finalize(buf, self._give, nbytes, ptr)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)

    def _give(self, nbytes: int, ptr: int) -> None:
        with self._lock:
            lst = self._free.setdefault(nbytes, [])
            if len(lst) < self.MAX_FREE_PER_SIZE:
                lst.append(ptr)
                return
        try:
            lib().epid_host_free(_P(ptr))
        except Exception:
            pass


_RESULT_POOL = _PinnedPool()


def frame_stats(ctx: Context, batch: Batch, view=None, percentiles=()):
    (n, h, w), _ = batch.shape_dtype
    r0, c0, vh, vw = view if view is not None else (0, 0, h, w)
    q = np.asarray(percentiles, dtype=np.float64)
    nq = q.size
    mn, mx, sm = np.empty(n), np.empty(n), np.empty(n)
    rows, cols = np.empty((n, vh)), np.empty((n, vw))
    pct = np.empty((n, max(nq, 1)))
    check(lib().epid_frame_stats(ctx.handle, batch.handle, r0, c0, vh, vw, _ptr(q) if nq else None, nq, _ptr(mn), _ptr(mx),
                                 _ptr(sm), _ptr(rows), _ptr(cols), _ptr(pct)))
    return {"min": mn, "max": mx, "sum": sm, "rowsum": rows, "colsum": cols, "percentiles": pct[:, :nq]}


def frame_histogram(ctx: Context, batch: Batch, view=None) -> np.ndarray:
    (n, h, w), _ = batch.shape_dtype
    r0, c0, vh, vw = view if view is not None else (0, 0, h, w)
    hist = np.empty((n, 65536), np.uint32)
    check(lib().epid_frame_histogram(ctx.handle, batch.handle, r0, c0, vh, vw, _ptr(hist)))
    return hist


def find_peaks(ctx: Context, values, threshold=-np.inf, peak_separation=0, max_number=None, fwxm_height=0.5, min_width=0,
               search_region=(0.0, 1.0), peak_sort="prominences", required_prominence=None):
    v = np.ascontiguousarray(values, dtype=np.float64)
    n = v.size
    p = PeakParams(float(threshold), float(peak_separation), int(max_number) if max_number else 0, float(fwxm_height),
                   float(min_width), float(search_region[0]), float(search_region[1]), 1 if peak_sort == "peak_heights" else 0,
                   -1.0 if required_prominence is None else float(required_prominence))
    cap = n // 2 + 2
    idx = np.empty(cap, np.int64)
    lb, rb = np.empty(cap, np.int64), np.empty(cap, np.int64)
    hts, prom, wid, wh, lip, rip = (np.empty(cap) for _ in range(6))
    cnt = C.c_int32()
    check(lib().epid_find_peaks(ctx.handle, _ptr(v), n, C.byref(p), cap, _ptr(idx), _ptr(hts), _ptr(prom), _ptr(lb), _ptr(rb),
                                _ptr(wid), _ptr(wh), _ptr(lip), _ptr(rip), C.byref(cnt)))
    c = cnt.value
    props = {"peak_heights": hts[:c].copy(), "prominences": prom[:c].copy(), "left_bases": lb[:c].copy(),
             "right_bases": rb[:c].copy(), "widths": wid[:c].copy(), "width_heights": wh[:c].copy(),
             "left_ips": lip[:c].copy(), "right_ips": rip[:c].copy()}
    return idx[:c].copy(), props


def pf_analyze(ctx: Context, frames, params: PFParams, meas_cap: int = 1024, host_pipeline: bool = False):
    """frames: a Batch (device-resident) or a uint16 ndarray [n,h,w] (host; chunked H2D overlapped with compute)."""
    if isinstance(frames, Batch):
        (n, _, _), _ = frames.shape_dtype
        summ = np.zeros(n, PF_SUMMARY_DTYPE)
        meas = np.zeros((n, meas_cap), PF_MEAS_DTYPE)
        check(lib().epid_pf_analyze(ctx.handle, frames.handle, C.byref(params), _ptr(summ), _ptr(meas), meas_cap))
        return summ, meas
    a = frames
    if a.dtype != np.uint16:
        raise TypeError("picket fence frames must be uint16")
    if a.ndim == 2:
        a = a[None]
    a = np.ascontiguousarray(a)
    n, h, w = a.shape
    # every element of both blocks is overwritten by the device-to-host copy of the (zero-initialised) device result arrays
    summ = _RESULT_POOL.take((n,), PF_SUMMARY_DTYPE)
    meas = _RESULT_POOL.take((n, meas_cap), PF_MEAS_DTYPE)
    check(lib().epid_pf_analyze_host(ctx.handle, _ptr(a), n, h, w, C.byref(params), _ptr(summ), _ptr(meas), meas_cap))
    return summ, meas


def pf_bench(ctx: Context, batch: Batch, params: PFParams, iters: int):
    total, stats = C.c_float(), C.c_float()
    launches = C.c_int64()
    check(lib().epid_pf_bench(ctx.handle, batch.handle, C.byref(params), iters, C.byref(total), C.byref(stats), C.byref(launches)))
    return total.value, stats.value, launches.value


PF_STAGE_NAMES = ("k_pf_init + k_pf_pilot", "k_pf_stream", "k_pf_tail", "k_pf_windows_fast", "k_pf_windows (generic)", "k_pf_finalize",
                  "exact front end (fallback)", "k_pf_win_medians", "k_pf_win_fwxm")


def pf_bench_timed(ctx: Context, batch: Batch, params: PFParams, iters: int):
    """(total_ms of `iters` passes, {stage name: ms per pass}, launches, frames re-run by the per-frame fallback)"""
    out = (C.c_float * 16)()
    total = C.c_float()
    launches, redone = C.c_int64(), C.c_int64()
    check(lib().epid_pf_bench_timed(ctx.handle, batch.handle, C.byref(params), iters, C.byref(total), out, 16, C.byref(launches),
                                    C.byref(redone)))
    return total.value, {name: out[k] / iters for k, name in enumerate(PF_STAGE_NAMES)}, launches.value, redone.value


def pf_bench_stages(ctx: Context, batch: Batch, params: PFParams, iters: int) -> dict:
    """{stage name: ms per pass} from CUDA events recorded between the kernels of `iters` device-resident passes."""
    return pf_bench_timed(ctx, batch, params, iters)[1]


def gaussian_kernel_table(max_sigma: int):
    """scipy/ndimage/_filters.py:_gaussian_kernel1d (order 0, truncate 4) for sigma = 1 .. max_sigma, concatenated.
    Host-side table of filter weights (the same numpy expression scipy evaluates); offsets[s] = start of sigma s."""
    offsets = np.zeros(max_sigma + 1, np.int32)
    chunks = []
    pos = 0
    for s in range(1, max_sigma + 1):
        sd = float(s)
        lw = int(4.0 * sd + 0.5)
        x = np.arange(-lw, lw + 1)
        phi = np.exp(-0.5 / (sd * sd) * x**2)
        w = (phi / phi.sum())[::-1]
        offsets[s] = pos
        chunks.append(np.ascontiguousarray(w, dtype=np.float64))
        pos += w.size
    return np.concatenate(chunks), offsets


def starshot_analyze(ctx: Context, frames, params: StarParams) -> np.ndarray:
    """frames: a Batch (device-resident, uint16) or a uint16 ndarray [n,h,w] / [h,w]; one STAR_RESULT_DTYPE row per frame."""
    own = None
    if not isinstance(frames, Batch):
        a = np.asarray(frames)
        if a.dtype != np.uint16:
            raise TypeError("starshot frames must be uint16")
        own = frames = Batch.upload(ctx, a)
    (n, h, w), _ = frames.shape_dtype
    # CollapsedCircleProfile length <= 2 pi * 1.1 * 0.95 * (dim / 2) * 3; sigma = round(0.003 * length)
    max_sigma = max(int(round(0.003 * (10 * max(h, w) + 64))) + 1, 2)
    gw, go = gaussian_kernel_table(max_sigma)
    res = np.zeros(n, STAR_RESULT_DTYPE)
    try:
        check(lib().epid_starshot_analyze(ctx.handle, frames.handle, C.byref(params), _ptr(gw), _ptr(go), max_sigma, _ptr(res)))
    finally:
        if own is not None:
            own.free()
    return res


def gaussian_kernel1d(sigma: float, truncate: float = 4.0):
    """scipy/ndimage/_filters.py:_gaussian_kernel1d (order 0), reversed as gaussian_filter1d hands it to correlate1d."""
    sd = float(sigma)
    lw = int(truncate * sd + 0.5)
    x = np.arange(-lw, lw + 1)
    phi = np.exp(-0.5 / (sd * sd) * x**2)
    return np.ascontiguousarray((phi / phi.sum())[::-1], dtype=np.float64), lw


def field_analyze(ctx: Context, frames, params: FieldParams) -> np.ndarray:
    """frames: a Batch (device-resident, uint16) or a uint16 ndarray [n,h,w] / [h,w]; one FIELD_RESULT_DTYPE row per frame."""
    own = None
    if not isinstance(frames, Batch):
        a = np.asarray(frames)
        if a.dtype != np.uint16:
            raise TypeError("field analysis frames must be uint16")
        own = frames = Batch.upload(ctx, a)
    (n, h, w), _ = frames.shape_dtype
    gh = gv = None
    lh = lv = 0
    if params.edge != 0:
        # gaussian_filter1d(values, sigma=edge_smoothing_ratio * len(values)) (core/profile.py:1655-1659): one table per profile length
        nh = lib().epid_field_profile_len(w, params.dpmm, params.interpolation, params.interpolation_resolution_mm)
        nv = lib().epid_field_profile_len(h, params.dpmm, params.interpolation, params.interpolation_resolution_mm)
        gh, lh = gaussian_kernel1d(params.edge_smoothing_ratio * nh)
        gv, lv = gaussian_kernel1d(params.edge_smoothing_ratio * nv)
    res = np.zeros(n, FIELD_RESULT_DTYPE)
    try:
        check(lib().epid_field_analyze(ctx.handle, frames.handle, C.byref(params), _ptr(gh), lh, _ptr(gv), lv, _ptr(res)))
    finally:
        if own is not None:
            own.free()
    return res


def wl2d_analyze(ctx: Context, frames, params: WlParams) -> np.ndarray:
    """frames: a Batch (device-resident, uint16) or a uint16 ndarray [n,h,w] / [h,w]; one WL_RESULT_DTYPE row per frame."""
    own = None
    if not isinstance(frames, Batch):
        a = np.asarray(frames)
        if a.dtype != np.uint16:
            raise TypeError("Winston-Lutz frames must be uint16")
        own = frames = Batch.upload(ctx, a)
    (n, _, _), _ = frames.shape_dtype
    res = np.zeros(n, WL_RESULT_DTYPE)
    try:
        check(lib().epid_wl2d_analyze(ctx.handle, frames.handle, C.byref(params), _ptr(res)))
    finally:
        if own is not None:
            own.free()
    return res


def _as_batch(ctx: Context, frames, dtypes=None):
    """-> (Batch, owned?) for a Batch or an ndarray [h,w] / [n,h,w]."""
    if isinstance(frames, Batch):
        return frames, False
    a = np.ascontiguousarray(frames)
    if a.ndim == 2:
        a = a[None]
    if dtypes is not None and a.dtype not in dtypes:
        raise TypeError(f"dtype {a.dtype} is not supported here")
    return Batch.upload(ctx, a), True


def disk_locate(ctx: Context, frames, params: DiskParams) -> np.ndarray:
    """SizedDiskRegion / SizedDiskLocator on uint16 frames: one DISK_RESULT_DTYPE row per frame."""
    b, own = _as_batch(ctx, frames, (np.dtype(np.uint16),))
    (n, _, _), _ = b.shape_dtype
    res = np.zeros(n, DISK_RESULT_DTYPE)
    try:
        check(lib().epid_disk_locate(ctx.handle, b.handle, C.byref(params), _ptr(res)))
    finally:
        if own:
            b.free()
    return res


def roi_stats(ctx: Context, frames, verts_xy) -> dict:
    """RectangleROI statistics: verts_xy [nroi, 4, 2] corner (x, y) -> dict of [n, nroi] arrays (count, mean, std, min, max)."""
    v = np.ascontiguousarray(verts_xy, dtype=np.float64).reshape(-1, 4, 2)
    b, own = _as_batch(ctx, frames)
    (n, _, _), _ = b.shape_dtype
    out = {k: np.empty((n, len(v))) for k in ("count", "mean", "std", "min", "max")}
    try:
        check(lib().epid_roi_stats(ctx.handle, b.handle, len(v), _ptr(v), _ptr(out["count"]), _ptr(out["mean"]), _ptr(out["std"]),
                                   _ptr(out["min"]), _ptr(out["max"])))
    finally:
        if own:
            b.free()
    return out


DISK_MAX_PCT = 16


def disk_roi_stats(ctx: Context, frames, centers_xy, radii, percentiles=()) -> dict:
    """DiskROI statistics of k disks (centers_xy [k, 2] as (x, y), radii [k]) on every frame -> dict of [n, k] arrays (count, mean, std,
    min, max, median) and "percentile" [n, k, p].  Empty disks give count 0 and NaN; IndexError for a disk over the bottom / right edge."""
    c = np.ascontiguousarray(centers_xy, dtype=np.float64).reshape(-1, 2)
    r = np.ascontiguousarray(np.broadcast_to(np.asarray(radii, dtype=np.float64), (len(c),)))
    q = np.ascontiguousarray([float(p) for p in np.atleast_1d(percentiles)], dtype=np.float64)
    if len(q) > DISK_MAX_PCT:
        raise ValueError(f"at most {DISK_MAX_PCT} percentiles per call")
    b, own = _as_batch(ctx, frames)
    (n, _, _), _ = b.shape_dtype
    out = {k: np.empty((n, len(c))) for k in ("count", "mean", "std", "min", "max", "median")}
    out["percentile"] = np.empty((n, len(c), len(q)))
    try:
        check(lib().epid_disk_roi_stats(ctx.handle, b.handle, len(c), _ptr(c), _ptr(r), len(q), _ptr(q) if len(q) else None,
                                        _ptr(out["count"]), _ptr(out["mean"]), _ptr(out["std"]), _ptr(out["min"]), _ptr(out["max"]),
                                        _ptr(out["median"]), _ptr(out["percentile"])))
    finally:
        if own:
            b.free()
    return out


def disk_roi_pixels(ctx: Context, frames, frame: int, center_xy, radius: float, clip: bool = False, indices: bool = False):
    """One disk's pixel values on frame ``frame`` in np.nonzero order (DiskROI.circle_mask; clip=True: the clipped pixel set of
    masked_array).  indices=True also returns skimage's (rows, cols)."""
    c = np.ascontiguousarray(center_xy, dtype=np.float64).reshape(2)
    b, own = _as_batch(ctx, frames)
    try:
        _, dt = b.shape_dtype
        n = C.c_int64()
        check(lib().epid_disk_roi_pixels(ctx.handle, b.handle, int(frame), _ptr(c), float(radius), int(bool(clip)), 0, None, None, None,
                                         C.byref(n)))
        vals = np.empty(n.value, dt)
        rows, cols = np.empty(n.value, np.int32), np.empty(n.value, np.int32)
        if n.value:
            check(lib().epid_disk_roi_pixels(ctx.handle, b.handle, int(frame), _ptr(c), float(radius), int(bool(clip)), n.value, _ptr(vals),
                                             _ptr(rows), _ptr(cols), C.byref(n)))
    finally:
        if own:
            b.free()
    return (vals, rows.astype(np.intp), cols.astype(np.intp)) if indices else vals


def vmat_analyze(ctx: Context, img1, img2, params: VmatParams) -> np.ndarray:
    """n (image 1, image 2) pairs of uint16 frames (Batch or ndarray [n,h,w] / [h,w]) -> one VMAT_RESULT_DTYPE row per pair."""
    b1, own1 = _as_batch(ctx, img1, (np.dtype(np.uint16),))
    try:
        b2, own2 = _as_batch(ctx, img2, (np.dtype(np.uint16),))
    except Exception:
        if own1:
            b1.free()
        raise
    (n, _, _), _ = b1.shape_dtype
    res = np.zeros(n, VMAT_RESULT_DTYPE)
    try:
        check(lib().epid_vmat_analyze(ctx.handle, b1.handle, b2.handle, C.byref(params), _ptr(res)))
    finally:
        if own1:
            b1.free()
        if own2:
            b2.free()
    return res


def divide(ctx: Context, num, den, sign_off=None) -> np.ndarray:
    """num / den as float64 (uint16 or float64 inputs of equal shape); sign_off [n, 2, 2] = (sign, offset) of num / den per frame."""
    a, b = np.ascontiguousarray(num), np.ascontiguousarray(den)
    squeeze = a.ndim == 2
    if a.dtype != b.dtype or a.dtype not in (np.uint16, np.float64):
        a, b = a.astype(np.float64), b.astype(np.float64)
    ba, bb = Batch.upload(ctx, a), Batch.upload(ctx, b)
    so = None if sign_off is None else np.ascontiguousarray(sign_off, dtype=np.float64).reshape(-1, 4)
    h = _P()
    try:
        check(lib().epid_divide(ctx.handle, ba.handle, bb.handle, _ptr(so), C.byref(h)))
        out = Batch(ctx, h)
        try:
            r = out.download()
        finally:
            out.free()
    finally:
        ba.free()
        bb.free()
    return r[0] if squeeze else r


def dlg_analyze(ctx: Context, frames, bottom, top, c0: int, c1: int, planned):
    """-> (measured [n, nleaf], slope [n], intercept [n], dlg [n]) for uint16 frames."""
    b, own = _as_batch(ctx, frames, (np.dtype(np.uint16),))
    (n, _, _), _ = b.shape_dtype
    bot = np.ascontiguousarray(bottom, dtype=np.int32)
    tp = np.ascontiguousarray(top, dtype=np.int32)
    pl = np.ascontiguousarray(planned, dtype=np.float64)
    nleaf = len(bot)
    meas, slope, icpt, dlg = np.empty((n, nleaf)), np.empty(n), np.empty(n), np.empty(n)
    try:
        check(lib().epid_dlg_analyze(ctx.handle, b.handle, nleaf, _ptr(bot), _ptr(tp), int(c0), int(c1), _ptr(pl), _ptr(meas), _ptr(slope),
                                     _ptr(icpt), _ptr(dlg)))
    finally:
        if own:
            b.free()
    return meas, slope, icpt, dlg


def global_locate(ctx: Context, frames, params: LocateParams, region_cap: int = 1024):
    """Whole-frame threshold sweep: -> list (per frame) of REGION_DTYPE arrays in the reference's visiting order."""
    b, own = _as_batch(ctx, frames, (np.dtype(np.uint16),))
    (n, _, _), _ = b.shape_dtype
    regs = np.zeros((n, region_cap), REGION_DTYPE)
    counts, flags = np.zeros(n, np.int32), np.zeros(n, np.int32)
    try:
        check(lib().epid_global_locate(ctx.handle, b.handle, C.byref(params), _ptr(regs), int(region_cap), _ptr(counts), _ptr(flags)))
    finally:
        if own:
            b.free()
    if (flags != 0).any():
        raise MemoryError(f"global locator: device lists overflowed (flags {flags.tolist()}); raise region_cap or pre-filter the frame")
    return [regs[i, : counts[i]].copy() for i in range(n)]


def canny(ctx: Context, image: np.ndarray, sigma: float = 1.0, low_threshold: float = 0.1, high_threshold: float = 0.2) -> np.ndarray:
    """skimage.feature.canny semantics for a float64 image [h, w] (or [n, h, w]) -> boolean edge map(s)."""
    a = np.ascontiguousarray(image, dtype=np.float64)
    squeeze = a.ndim == 2
    w, lw = gaussian_kernel1d(float(sigma))
    b = Batch.upload(ctx, a)
    h = _P()
    try:
        check(lib().epid_canny(ctx.handle, b.handle, _ptr(w), int(lw), float(low_threshold), float(high_threshold), C.byref(h)))
        out = Batch(ctx, h)
        try:
            r = out.download()
        finally:
            out.free()
    finally:
        b.free()
    r = r.astype(bool)
    return r[0] if squeeze else r


def hough_line(ctx: Context, edges: np.ndarray, theta: np.ndarray):
    """skimage.transform.hough_line: -> (accumulator Batch [1, 2 * offset + 1, ntheta] int32 on the device, offset)"""
    e = np.ascontiguousarray(edges).astype(np.uint8)
    th = np.ascontiguousarray(theta, dtype=np.float64)
    b = Batch.upload(ctx, e)
    h, off = _P(), C.c_int32()
    try:
        check(lib().epid_hough_line(ctx.handle, b.handle, len(th), _ptr(th), C.byref(h), C.byref(off)))
    finally:
        b.free()
    return Batch(ctx, h), off.value


def hough_candidates(ctx: Context, accum: Batch, min_xdistance: int, min_ydistance: int, threshold: float | None = None, cap: int = 1 << 16):
    """-> (candidates [k, 3] (row, col, value), global maximum, max-filtered accumulator Batch)"""
    cand = np.zeros((cap, 3), np.int32)
    cnt, gmax = C.c_int32(), C.c_int32()
    h = _P()
    check(lib().epid_hough_candidates(ctx.handle, accum.handle, int(min_xdistance), int(min_ydistance), -1.0 if threshold is None else float(threshold),
                                      cap, _ptr(cand), C.byref(cnt), C.byref(gmax), C.byref(h)))
    return cand[: cnt.value].copy(), gmax.value, Batch(ctx, h)


def gather_i32(ctx: Context, img: Batch, yx: np.ndarray) -> np.ndarray:
    pts = np.ascontiguousarray(yx, dtype=np.int32).reshape(-1, 2)
    out = np.zeros(len(pts), np.int32)
    check(lib().epid_gather_i32(ctx.handle, img.handle, len(pts), _ptr(pts), _ptr(out)))
    return out


def weighted_centroid(ctx: Context, frames):
    """(cx, cy, total) arrays of length n: sum(x * a) / sum(a), sum(y * a) / sum(a), sum(a)."""
    b, own = _as_batch(ctx, frames)
    (n, _, _), _ = b.shape_dtype
    cx, cy, tot = np.empty(n), np.empty(n), np.empty(n)
    try:
        check(lib().epid_weighted_centroid(ctx.handle, b.handle, _ptr(cx), _ptr(cy), _ptr(tot)))
    finally:
        if own:
            b.free()
    return cx, cy, tot


def circle_profile(ctx: Context, image: np.ndarray, center, radius: float, start_angle: float = 0.0, ccw: bool = True,
                   sampling_ratio: float = 1.0, collapsed: bool = False, width_ratio: float = 0.1, num_profiles: int = 20):
    """(profile, x_locations, y_locations) of a CircleProfile / CollapsedCircleProfile of one image."""
    a = np.ascontiguousarray(image)
    if a.dtype not in (np.uint8, np.uint16, np.float32, np.float64):
        a = a.astype(np.float64)
    b = Batch.upload(ctx, a)
    rmax = radius * (1 + width_ratio) if collapsed else radius
    cap = int(np.ceil(2 * np.pi * rmax * sampling_ratio)) + 8
    prof, xl, yl = np.empty(cap), np.empty(cap), np.empty(cap)
    cnt = C.c_int32()
    try:
        check(lib().epid_circle_profile(ctx.handle, b.handle, float(center[0]), float(center[1]), float(radius), float(start_angle),
                                        1 if ccw else 0, float(sampling_ratio), 1 if collapsed else 0, float(width_ratio),
                                        int(num_profiles), cap, _ptr(prof), _ptr(xl), _ptr(yl), C.byref(cnt)))
    finally:
        b.free()
    c = cnt.value
    return prof[:c].copy(), xl[:c].copy(), yl[:c].copy()


def single_profile(ctx: Context, values, params: SpParams, *, fwxm_x=50.0, penumbra=(20.0, 80.0), in_field_ratio=0.8,
                   slope_exclusion_ratio=0.2, x_values=None):
    """SingleProfile(values, ...) + every query method in one launch -> (result row, values, field values)."""
    v = np.ascontiguousarray(values, dtype=np.float64)
    n0 = v.size
    if params.interpolation == 1:
        n = int(round(n0 / (params.dpmm * params.interpolation_resolution_mm))) if params.dpmm > 0 else int(round(n0 * params.interpolation_factor))
    else:
        n = n0
    gw, lw = (gaussian_kernel1d(params.edge_smoothing_ratio * n) if params.edge == 1 else (None, 0))
    res = np.zeros(1, SP_RESULT_DTYPE)
    cap = n + 8
    vals, fv = np.empty(cap), np.empty(cap)
    xv = None if x_values is None else np.ascontiguousarray(x_values, dtype=np.float64)
    if xv is not None and xv.size != n0:
        raise ValueError("x_values and values must have the same length")
    check(lib().epid_single_profile(ctx.handle, _ptr(v), _ptr(xv), n0, C.byref(params), _ptr(gw), lw, n, float(fwxm_x), float(penumbra[0]),
                                    float(penumbra[1]), float(in_field_ratio), float(slope_exclusion_ratio), _ptr(res), _ptr(vals),
                                    _ptr(fv), cap))
    r = res[0]
    return r, vals[: int(r["n"])].copy(), fv[: int(r["fd_field_values_n"])].copy()
