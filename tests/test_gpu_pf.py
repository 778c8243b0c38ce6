"""GPU parity: PicketFence pipeline in CUDA (through the C-ABI) vs the committed reference goldens and the oracle port.

Bars (BASELINE.json north_star): bit-exact for orientation, picket indices, leaf / picket / kiss counts, pass flags;
<= 0.01 px for sub-pixel positions (we assert 1e-6 px; the fp64 profile arithmetic mirrors scipy's operation order)."""
import warnings

import numpy as np
import pytest

from tests.golden.pf_cases import CASES, case_frame

pytestmark = pytest.mark.gpu

GOLD = np.load("tests/golden/pf_golden.npz")
POS_TOL_PX = 1e-6     # required: 0.01 px
ERR_TOL_MM = 1e-6


def gpu_run(name):
    from pylinac_b200 import picketfence as pf

    a, ps, sid, ck, ak = case_frame(name)
    dpmm = (1 / ps) * sid / 1000.0
    ck = dict(ck)
    if ck.get("mlc") == "HD":
        ck["mlc"] = pf.MLC.HD_MILLENNIUM
    res = pf.analyze_batch(a[None], dpmm, **ck, **ak)
    return res[0], dpmm


def _compare_with_golden(r, name, GOLD):
    if f"{name}/raises" in GOLD:
        assert r.status != 0
        with pytest.raises(ValueError):
            r.raise_for_status()
        return
    assert r.status == 0, r.status
    g = lambda k: GOLD[f"{name}/{k}"]
    s = r.s
    # ---- bit-exact integers
    assert int(s["orientation"]) == int(g("orientation"))
    assert int(s["n_pickets"]) == int(g("number_of_pickets"))
    assert int(s["n_meas"]) == int(g("n_meas"))
    assert tuple(int(v) for v in (s["height"], s["width"])) == tuple(int(v) for v in g("shape"))
    # the golden stores the set of picket indices that produced measurements (sorted)
    assert sorted(int(v) for v in r.picket_idx) == [int(v) for v in g("picket_idx")]
    assert np.array_equal(r.m["leaf_num"], g("meas_leaf"))
    assert np.array_equal(r.m["picket"], g("meas_picket"))
    assert bool(s["passed"]) == bool(g("passed"))
    if float(g("max_error")) > 10 * ERR_TOL_MM:
        # on the reference's noise-free "perfect" fixtures every error is rounding noise (~1e-13 mm): which picket / leaf holds
        # the largest of them is decided below the fp tolerance and is not a parity property
        assert int(s["max_error_picket"]) == int(g("max_error_picket"))
        assert str(r.max_error_leaf) == str(g("max_error_leaf"))
    assert [str(x) for x in r.failed_leaves()] == [str(x) for x in g("failed_leaves")]
    # ---- sub-pixel quantities
    npos = g("meas_position").shape[1]
    np.testing.assert_allclose(r.m["position"][:, :npos], g("meas_position"), rtol=0, atol=POS_TOL_PX)
    np.testing.assert_allclose(r.m["error"][:, :npos], g("meas_error"), rtol=0, atol=ERR_TOL_MM)
    np.testing.assert_allclose(r.m["width_mm"], g("meas_width_mm"), rtol=0, atol=ERR_TOL_MM)
    npk = int(s["n_pickets"])
    np.testing.assert_allclose(s["picket_spacing_px"], g("picket_spacing"), rtol=0, atol=0)
    fits = np.stack([s["fit_slope"][:npk], s["fit_intercept"][:npk]], axis=1)
    np.testing.assert_allclose(fits[:, 0], g("fits")[:, 0], rtol=0, atol=1e-9)
    np.testing.assert_allclose(fits[:, 1], g("fits")[:, 1], rtol=0, atol=POS_TOL_PX)
    np.testing.assert_allclose(s["offsets_from_cax_mm"][:npk], g("offsets_from_cax_mm"), rtol=0, atol=ERR_TOL_MM)
    for key, gk in [("percent_passing", "percent_passing"), ("max_error_mm", "max_error"), ("abs_median_error_mm", "abs_median_error"),
                    ("mean_picket_spacing_mm", "mean_picket_spacing"), ("mlc_skew", "mlc_skew")]:
        np.testing.assert_allclose(float(s[key]), float(g(gk)), rtol=0, atol=ERR_TOL_MM, err_msg=key)
    pw = np.stack([s["picket_width_max"][:npk], s["picket_width_mean"][:npk], s["picket_width_median"][:npk], s["picket_width_min"][:npk]], axis=1)
    np.testing.assert_allclose(pw, g("picket_widths"), rtol=0, atol=ERR_TOL_MM)


@pytest.mark.parametrize("name", CASES)
def test_pf_matches_reference_golden(name):
    r, dpmm = gpu_run(name)
    _compare_with_golden(r, name, GOLD)


def _docs_names():
    from tests.golden import pf_docs_cases as dc

    return list(dc.DOCS)


@pytest.mark.parametrize("name", _docs_names())
def test_pf_matches_reference_on_docs_fixture(name):
    """The reference's own fixtures (docs/source/files/*.dcm, 1280 x 1280) with the docs recipes' analyze() arguments."""
    from pylinac_b200 import picketfence as pf
    from tests.golden import pf_docs_cases as dc

    a, ps, sid, ak = dc.docs_frame(name)
    r = pf.analyze_batch(a[None], (1 / ps) * sid / 1000.0, **ak)[0]
    _compare_with_golden(r, name, np.load("tests/golden/pf_docs_golden.npz"))


def test_pf_batch_matches_oracle_and_is_frame_independent():
    """A mixed batch: every frame's result equals its single-frame result and the oracle's."""
    from oracle import pf_oracle, synth
    from pylinac_b200 import picketfence as pf

    frames = np.stack([synth.bench_pf_frame(i) for i in range(20, 26)])
    res = pf.analyze_batch(frames, 2.56)
    for i in range(len(frames)):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            o = pf_oracle.pf_analyze(frames[i], 2.56)
        r = res[i]
        assert r.status == 0
        assert np.array_equal(np.sort(r.picket_idx), np.sort(o["picket_idx"]))
        assert int(r.s["n_meas"]) == o["n_meas"]
        np.testing.assert_allclose(r.m["position"][:, :1], o["meas_position"], rtol=0, atol=POS_TOL_PX)
        np.testing.assert_allclose(r.m["error"][:, :1], o["meas_error"], rtol=0, atol=ERR_TOL_MM)
        single = pf.analyze_batch(frames[i][None], 2.56)[0]
        assert np.array_equal(single.m["position"], r.m["position"])


def test_pf_host_pipeline_equals_device_resident():
    from oracle import synth
    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    frames = np.stack([synth.bench_pf_frame(i) for i in range(40, 43)] * 30)  # 90 frames -> several chunks
    ctx = nat.Context.default()
    params = pf.make_params(2.56, frames.shape[1:])
    s1, m1 = nat.pf_analyze(ctx, frames, params)
    b = nat.Batch.upload(ctx, frames)
    s2, m2 = nat.pf_analyze(ctx, b, params)
    b.free()
    assert np.array_equal(s1["picket_idx"], s2["picket_idx"])
    assert np.array_equal(s1["n_meas"], s2["n_meas"])
    for i in range(len(frames)):   # rows beyond n_meas are unspecified
        k = int(s1["n_meas"][i])
        assert k == 500
        assert np.array_equal(m1["position"][i, :k], m2["position"][i, :k])
        assert np.array_equal(m1["error"][i, :k], m2["error"][i, :k])
    assert np.array_equal(s1["max_error_mm"], s2["max_error_mm"])


def test_picketfence_class_api():
    from oracle import synth
    from pylinac_b200.picketfence import MLC, Orientation, PicketFence

    a = synth.bench_pf_frame(0)
    pfo = PicketFence(a, image_kwargs={"dpi": 25.4 / 0.390625, "sid": 1000})
    pfo.analyze()
    assert pfo.num_pickets == 10
    assert pfo.orientation == Orientation.UP_DOWN
    assert pfo.passed
    rd = pfo.results_data()
    assert rd.number_of_pickets == 10
    assert abs(rd.max_error_mm - float(GOLD["bench0/max_error"])) < 1e-6
    assert len(rd.mlc_positions_by_leaf) == 50
    assert "Picket Fence Results" in pfo.results()
    assert len(pfo.mlc_meas) == 500 and len(pfo.pickets) == 10
    d = pfo.results_data(as_dict=True)
    assert d["percent_leaves_passing"] == 100.0


def _variants():
    """Adversarial inputs for the sample-guided selection of the fused front kernel."""
    from oracle import synth

    out = {}
    a = synth.bench_pf_frame(11)
    out["plain"] = (a, {})
    out["crop5_misaligned"] = (a, {"crop_mm": 2})                       # 5 px crop: the view is not 16-byte aligned
    out["crop0"] = (a, {"crop_mm": 0})
    out["quantised_8bit"] = ((a >> 8) << 8, {})                         # 256 heavy values
    out["saturated"] = (np.minimum(a.astype(np.uint32) * 2, 65535).astype(np.uint16), {})   # clipped ceiling
    out["offset_floor"] = ((a // 2 + 20000).astype(np.uint16), {})      # heavy floor value that is not zero
    out["left_right"] = (np.ascontiguousarray(a.T), {})
    out["inverted"] = ((a.max() - a).astype(np.uint16), {})
    rng = np.random.default_rng(3)
    out["strong_noise"] = (np.clip(a.astype(np.int64) + rng.normal(0, 1500, a.shape), 0, 65535).astype(np.uint16), {})
    out["given_orientation"] = (a, {"orientation": "Up-Down"})
    return out


@pytest.mark.parametrize("name", list(_variants()))
def test_fast_front_kernel_equals_exact_pipeline(name):
    """The fused sample-guided front kernel must give bit-identical results to the exact-histogram pipeline
    (which is pinned to the reference by the golden tests above), whichever path ends up being used."""
    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    a, kw = _variants()[name]
    frames = np.stack([a, a[::-1].copy(), a])
    ctx = nat.Context.default()
    try:
        ctx.set_option(nat.OPT_PF_EXACT_ONLY, 1)
        exact = pf.analyze_batch(frames, 2.56, **kw)
        ctx.set_option(nat.OPT_PF_EXACT_ONLY, 0)
        fast = pf.analyze_batch(frames, 2.56, **kw)
    finally:
        ctx.set_option(nat.OPT_PF_EXACT_ONLY, 0)
    for k in exact.summary.dtype.names:
        np.testing.assert_array_equal(exact.summary[k], fast.summary[k], err_msg=k)
    for i in range(len(frames)):
        if int(exact.summary["status"][i]) == 0:
            m = int(exact.summary["n_meas"][i])
            for k in exact.meas.dtype.names:
                np.testing.assert_array_equal(exact.meas[k][i, :m], fast.meas[k][i, :m], err_msg=k)


def test_fast_front_kernel_is_used_for_the_benchmark_frames():
    from oracle import synth
    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    ctx = nat.Context.default()
    before = ctx.counter(nat.CTR_PF_FALLBACKS)
    frames = np.stack([synth.bench_pf_frame(i) for i in range(60, 66)])
    res = pf.analyze_batch(frames, 2.56)
    assert all(int(s) == 0 for s in res.summary["status"])
    assert ctx.counter(nat.CTR_PF_FALLBACKS) == before, "the fused front kernel fell back to the exact pipeline"


def _shape_cases():
    """Non-square / odd-sized EPID panels: aS500 (384 x 512), aS1000 (768 x 1024), and views whose rows are not a multiple
    of 8 pixels (unaligned pitch: the TMA front end declines them and the exact pipeline runs)."""
    from oracle import synth

    out = {}
    fr = synth.as1000(1000.0)
    out["as1000_768x1024"] = (synth.picketfence_frame(fr, pickets=7, picket_spacing_mm=25, picket_width_mm=3, seed=201), fr.pixel_size, 1000.0, {})
    fr = synth.as500(1000.0)
    out["as500_384x512"] = (synth.picketfence_frame(fr, pickets=5, picket_spacing_mm=30, picket_width_mm=4, picket_height_mm=200, seed=202),
                            fr.pixel_size, 1000.0, {})
    fr = synth.as1000(1000.0)
    a = synth.picketfence_frame(fr, pickets=7, picket_spacing_mm=25, picket_width_mm=3, orientation="left_right", seed=203)
    out["as1000_left_right"] = (a, fr.pixel_size, 1000.0, {})
    fr = synth.epid1024()
    a = synth.picketfence_frame(fr, seed=204)
    out["odd_1001x1019"] = (np.ascontiguousarray(a[11:1012, 3:1022]), fr.pixel_size, 1000.0, {})
    out["odd_1019x1001_crop0"] = (np.ascontiguousarray(a[3:1022, 11:1012]), fr.pixel_size, 1000.0, {"crop_mm": 0})
    return out


@pytest.mark.parametrize("name", list(_shape_cases()))
def test_pf_ragged_shapes_match_the_oracle(name):
    from oracle import pf_oracle
    from pylinac_b200 import picketfence as pf

    a, ps, sid, kw = _shape_cases()[name]
    dpmm = (1 / ps) * sid / 1000.0
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        o = pf_oracle.pf_analyze(a, dpmm, **kw)
    r = pf.analyze_batch(np.stack([a, a]), dpmm, **kw)[1]
    assert r.status == 0
    assert int(r.s["orientation"]) == int(o["orientation"])
    assert tuple(int(v) for v in (r.s["height"], r.s["width"])) == tuple(o["shape"])
    assert sorted(int(v) for v in r.picket_idx) == sorted(int(v) for v in o["picket_idx"])
    assert int(r.s["n_meas"]) == o["n_meas"] and o["n_meas"] > 50
    assert np.array_equal(r.m["leaf_num"], o["meas_leaf"]) and np.array_equal(r.m["picket"], o["meas_picket"])
    np.testing.assert_allclose(r.m["position"][:, :1], o["meas_position"], rtol=0, atol=POS_TOL_PX)
    np.testing.assert_allclose(r.m["error"][:, :1], o["meas_error"], rtol=0, atol=ERR_TOL_MM)
    np.testing.assert_allclose(float(r.s["max_error_mm"]), float(o["max_error"]), rtol=0, atol=ERR_TOL_MM)


def test_pf_degenerate_inputs_fail_like_the_reference():
    """Flat frames and frames without pickets raise ValueError in the reference (picketfence.py:760-764, 804-807); a batch
    keeps going and reports them per frame."""
    from oracle import synth
    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    good = synth.bench_pf_frame(70)
    flat = np.full_like(good, 1234)
    noise = np.random.default_rng(9).integers(1000, 1100, good.shape).astype(np.uint16)
    res = pf.analyze_batch(np.stack([good, flat, noise, good]), 2.56)
    assert res[0].status == 0 and res[3].status == 0
    assert np.array_equal(res[0].m["position"], res[3].m["position"])
    for k in (1, 2):
        assert res[k].status != 0
        with pytest.raises(ValueError):
            res[k].raise_for_status()
    with pytest.raises((ValueError, nat.NativeError)):
        pf.analyze_batch(np.zeros((1, 8, 8), np.uint16), 2.56)
    with pytest.raises(TypeError):
        pf.analyze_batch(np.zeros((1, 1024, 1024), np.float32), 2.56)


def _window_cases():
    from oracle import synth
    from tests.golden import pf_docs_cases as dc

    out = {}
    out["bench"] = (np.stack([synth.bench_pf_frame(i) for i in range(80, 86)]), 2.56, {})
    a = synth.bench_pf_frame(86)
    out["sag"] = (a[None], 2.56, {"sag_adjustment": 1.5})
    out["separate"] = (a[None], 2.56, {"separate_leaves": True, "nominal_gap_mm": 3})
    out["inverted"] = ((a.max() - a).astype(np.uint16)[None], 2.56, {})
    out["crop2_misaligned"] = (a[None], 2.56, {"crop_mm": 2})
    out["crop0"] = (a[None], 2.56, {"crop_mm": 0})
    out["wide_windows"] = (a[None], 2.56, {"leaf_analysis_width_ratio": 0.9, "picket_spacing": 40.0})
    for nm in ("as1200", "hdmlc", "fwxm70_edge", "tight_tol", "dead_pixel"):
        fr, ps, sid, ck, ak = case_frame(nm)
        ck = dict(ck)
        if ck.get("mlc") == "HD":
            from pylinac_b200 import picketfence as pf

            ck["mlc"] = pf.MLC.HD_MILLENNIUM
        out[nm] = (fr[None], (1 / ps) * sid / 1000.0, {**ck, **ak})
    for nm in ("rotated_up_down", "erroneous_leaves"):
        fr, ps, sid, ak = dc.docs_frame(nm)
        out["docs_" + nm] = (fr[None], (1 / ps) * sid / 1000.0, ak)
    return out


def test_pf_host_pipeline_staged_and_direct_result_paths_agree():
    """epid_pf_analyze_host DMA's the results straight into page-locked caller buffers and goes through its pinned staging area
    for pageable ones (a C caller's malloc'd arrays): both paths must deliver identical bytes for the used rows."""
    import ctypes as C

    from oracle import synth
    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    frames = np.ascontiguousarray(np.stack([synth.bench_pf_frame(i) for i in range(90, 93)] * 50))     # 150 frames: 3 chunks
    ctx = nat.Context.default()
    params = pf.make_params(2.56, frames.shape[1:])
    n, h, w = frames.shape
    cap = 1024
    s_direct, m_direct = nat.pf_analyze(ctx, frames, params, meas_cap=cap)                              # pooled pinned arrays
    s_staged = np.zeros(n, nat.PF_SUMMARY_DTYPE)                                                        # pageable
    m_staged = np.zeros((n, cap), nat.PF_MEAS_DTYPE)
    nat.check(nat.lib().epid_pf_analyze_host(ctx.handle, frames.ctypes.data_as(C.c_void_p), n, h, w, C.byref(params),
                                             s_staged.ctypes.data_as(C.c_void_p), m_staged.ctypes.data_as(C.c_void_p), cap))
    assert (s_direct["status"] == 0).all()
    for k in s_direct.dtype.names:
        np.testing.assert_array_equal(s_direct[k], s_staged[k], err_msg=k)
    for i in range(n):
        m = int(s_direct["n_meas"][i])
        for k in m_direct.dtype.names:
            np.testing.assert_array_equal(m_direct[k][i, :m], m_staged[k][i, :m], err_msg=k)


@pytest.mark.parametrize("name", list(_window_cases()))
def test_two_kernel_window_path_equals_per_window_kernel(name):
    """The default window path (k_pf_win_medians + k_pf_win_fwxm, pf_windows2.cu) must reproduce the single per-window kernel
    (k_pf_windows_fast, pinned to the reference by the golden tests) bit for bit, on frames it covers and on frames it declines."""
    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    frames, dpmm, kw = _window_cases()[name]
    ctx = nat.Context.default()
    try:
        ctx.set_option(nat.OPT_PF_WIN2, 0)
        old = pf.analyze_batch(frames, dpmm, **kw)
        ctx.set_option(nat.OPT_PF_WIN2, 1)
        new = pf.analyze_batch(frames, dpmm, **kw)
    finally:
        ctx.set_option(nat.OPT_PF_WIN2, 1)
    for k in old.summary.dtype.names:
        np.testing.assert_array_equal(old.summary[k], new.summary[k], err_msg=k)
    for i in range(len(frames)):
        if int(old.summary["status"][i]) == 0:
            m = int(old.summary["n_meas"][i])
            assert m > 0
            for k in old.meas.dtype.names:
                np.testing.assert_array_equal(old.meas[k][i, :m], new.meas[k][i, :m], err_msg=k)


def test_two_kernel_window_path_runs_for_the_benchmark_frames():
    from oracle import synth
    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    ctx = nat.Context.default()
    frames = np.stack([synth.bench_pf_frame(i) for i in range(60, 76)])
    b = nat.Batch.upload(ctx, frames)
    try:
        st = nat.pf_bench_stages(ctx, b, pf.make_params(2.56, frames.shape[1:]), 2)
    finally:
        b.free()
    assert st["k_pf_win_medians"] > 5 * st["k_pf_windows_fast"] > 0, st
    # every kernel of the default pipeline is charged to its own stage, and only those
    assert {k for k, v in st.items() if v > 0} == {"k_pf_init + k_pf_pilot", "k_pf_stream", "k_pf_tail", "k_pf_windows_fast",
                                                   "k_pf_windows (generic)", "k_pf_finalize", "k_pf_win_medians", "k_pf_win_fwxm"}, st


def test_retired_pf_options_are_rejected():
    from pylinac_b200 import _native as nat

    ctx = nat.Context.default()
    for key in (2, 4, 6):       # retired option keys
        with pytest.raises(ValueError):
            ctx.set_option(key, 1)


def test_pf_mixed_batch_matches_the_oracle_frame_by_frame():
    """Certifiable, noisy (salt-and-pepper -> _check_for_noise median passes), inverted, left-right, flat and pattern-free frames
    interleaved in ONE batch: every frame must equal the oracle's result for that frame alone, whichever front end (certified
    stream kernel or exact per-frame re-run) and whichever window kernel ended up processing it."""
    from oracle import pf_oracle, synth
    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    rng = np.random.default_rng(77)
    base = [synth.bench_pf_frame(i) for i in range(300, 312)]
    frames, kinds = [], []
    for i, a in enumerate(base):
        kind = ("clean", "noisy", "inverted", "clean", "noisy2", "left_right", "flat", "clean", "noise_only", "noisy", "clean", "inverted")[i]
        if kind == "noisy":          # hot pixels: max > 1.25 p99.5 -> one median pass (picketfence.py:221-238)
            a = (a // 2).copy()
            idx = rng.integers(0, a.size, 40)
            a.ravel()[idx] = 65535
        elif kind == "noisy2":       # a 3 x 3 block of hot pixels survives two 3x3 median passes: three passes in the reference
            a = (a // 2).copy()
            a[500:503, 100:103] = 65535
            a[40, 40] = 65535
        elif kind == "inverted":
            a = (int(a.max()) - a.astype(np.int64)).astype(np.uint16)
        elif kind == "left_right":
            a = np.ascontiguousarray(a.T)
        elif kind == "flat":
            a = np.full_like(a, 777)
        elif kind == "noise_only":
            a = rng.integers(1000, 1100, a.shape).astype(np.uint16)
        frames.append(a)
        kinds.append(kind)
    frames = np.stack(frames)
    ctx = nat.Context.default()
    redone0 = ctx.counter(nat.CTR_PF_REDONE_FRAMES)
    res = pf.analyze_batch(frames, 2.56)
    redone = ctx.counter(nat.CTR_PF_REDONE_FRAMES) - redone0
    assert 0 < redone < len(frames), f"per-frame fallback expected for the noisy frames only, {redone} frames were re-run"
    n_noise = 0
    for i, kind in enumerate(kinds):
        r = res[i]
        try:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                o = pf_oracle.pf_analyze(frames[i], 2.56)
        except (ValueError, IndexError):
            assert r.status != 0, (i, kind)
            continue
        assert r.status == 0, (i, kind, r.status)
        n_noise += int(o["noise_median_passes"] > 0)
        assert int(r.s["noise_median_passes"]) == o["noise_median_passes"], (i, kind)
        assert int(r.s["orientation"]) == int(o["orientation"])
        assert sorted(int(v) for v in r.picket_idx) == sorted(int(v) for v in o["picket_idx"]), (i, kind)
        assert int(r.s["n_meas"]) == o["n_meas"], (i, kind)
        assert np.array_equal(r.m["leaf_num"], o["meas_leaf"]) and np.array_equal(r.m["picket"], o["meas_picket"])
        np.testing.assert_allclose(r.m["position"][:, :1], o["meas_position"], rtol=0, atol=POS_TOL_PX, err_msg=f"{i} {kind}")
        np.testing.assert_allclose(r.m["error"][:, :1], o["meas_error"], rtol=0, atol=ERR_TOL_MM, err_msg=f"{i} {kind}")
        np.testing.assert_allclose(float(r.s["max_error_mm"]), float(o["max_error"]), rtol=0, atol=ERR_TOL_MM)
    assert n_noise >= 2, "the mixed batch should contain frames that trigger the reference's noise filter"


def _mixed_frames(seed=5, n=96):
    """Benchmark frames with every 8th frame noisy: hot pixels (one median pass), every 24th with a hot 3 x 3 block (three passes)."""
    from oracle import synth

    rng = np.random.default_rng(seed)
    uniq = [synth.bench_pf_frame(i) for i in range(400, 408)]
    frames = np.stack([uniq[i % 8] for i in range(n)])
    kinds = []
    for i in range(n):
        if i % 24 == 7:
            a = frames[i] // 2
            a[500:503, 100:103] = 65535
            a[40, 40] = 65535
            frames[i] = a
            kinds.append("block")
        elif i % 8 == 3:
            a = frames[i] // 2
            a.ravel()[rng.integers(0, a.size, 40)] = 65535
            frames[i] = a
            kinds.append("hot")
        else:
            kinds.append("clean")
    return frames, kinds


def _assert_same_results(a, b):
    (sa, ma), (sb, mb) = a, b
    for k in sa.dtype.names:
        np.testing.assert_array_equal(sa[k], sb[k], err_msg=k)
    for i in range(len(sa)):
        m = int(sa["n_meas"][i])
        for k in ma.dtype.names:
            np.testing.assert_array_equal(ma[k][i, :m], mb[k][i, :m], err_msg=f"{k} frame {i}")


def test_pf_certified_noise_rerun_equals_the_exact_rerun():
    """The per-frame fallback: frames whose _has_noise() the single exact count certifies are median filtered and re-run by the
    certified fast pipeline (frames with a hot block are deferred again -> exact pipeline).  Every variant -- fast / exact re-run,
    device-resident (overlapped with the batch on the second stream) or host entry point -- must return bit-identical rows, and the
    hot-pixel frames must equal the oracle."""
    from oracle import pf_oracle
    from pylinac_b200 import _native as nat
    from pylinac_b200 import picketfence as pf

    frames, kinds = _mixed_frames()
    ctx = nat.Context.default()
    params = pf.make_params(2.56, frames.shape[1:])
    b = nat.Batch.upload(ctx, frames)
    results = {}
    counts = {}
    try:
        for fast_redo in (1, 0):
            ctx.set_option(nat.OPT_PF_FAST_REDO, fast_redo)
            r0, e0 = ctx.counter(nat.CTR_PF_REDONE_FRAMES), ctx.counter(nat.CTR_PF_EXACT_FRAMES)
            results[(fast_redo, "dev")] = nat.pf_analyze(ctx, b, params)
            counts[fast_redo] = (ctx.counter(nat.CTR_PF_REDONE_FRAMES) - r0, ctx.counter(nat.CTR_PF_EXACT_FRAMES) - e0)
            s, m = nat.pf_analyze(ctx, frames, params)
            results[(fast_redo, "host")] = (s.copy(), m.copy())
    finally:
        ctx.set_option(nat.OPT_PF_FAST_REDO, 1)
        b.free()
    n_hot, n_block = kinds.count("hot"), kinds.count("block")
    assert n_hot >= 8 and n_block >= 4
    assert counts[1] == (n_hot + n_block, n_block), counts      # only the hot-block frames need the exact pipeline
    assert counts[0] == (n_hot + n_block, n_hot + n_block), counts
    ref = results[(0, "dev")]
    for key, val in results.items():
        _assert_same_results(ref, val)
    s, m = ref
    assert np.all(s["status"] == 0)
    for i, kind in enumerate(kinds):
        assert int(s["noise_median_passes"][i]) == {"clean": 0, "hot": 1, "block": 3}[kind], (i, kind)
    for i in [kinds.index("hot"), kinds.index("block"), len(kinds) - 1 - kinds[::-1].index("hot")]:
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            o = pf_oracle.pf_analyze(frames[i], 2.56)
        nm = int(s["n_meas"][i])
        assert nm == o["n_meas"] and int(s["noise_median_passes"][i]) == o["noise_median_passes"]
        np.testing.assert_allclose(m["position"][i, :nm, :1], o["meas_position"], rtol=0, atol=POS_TOL_PX)


@pytest.mark.parametrize("name", ["noisy_wide_gap_up_down", "offset_picket", "perfect_left_right"])
def test_picketfence_reads_the_reference_dicom_files(name, tmp_path):
    """File -> pylinac_b200.dicom -> LinacDicomImage -> PicketFence(path).analyze(): the reference's docs fixtures end to end (the
    array is float64 after the identity rescale, like pydicom's; dpmm comes from ImagePlanePixelSpacing x RTImageSID / SAD)."""
    from pylinac_b200.picketfence import PicketFence
    from tests.golden import pf_docs_cases as dc

    p = tmp_path / (name + ".dcm")
    p.write_bytes(dc.docs_dcm_bytes(name))
    _, ps, sid, ak = dc.docs_frame(name)
    pfo = PicketFence(str(p))
    assert pfo._raw.array.dtype == np.float64 and pfo._raw.dpmm == pytest.approx((1 / ps) * sid / 1000.0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        pfo.analyze(**ak)
    _compare_with_golden(pfo._result, name, np.load("tests/golden/pf_docs_golden.npz"))
    assert "Gantry Angle" in pfo.results()


def test_analyze_files_equals_the_per_file_objects(tmp_path):
    """f1 ingest: picketfence.analyze_files (header parse + pixel bytes straight into page-locked memory + one batched analysis) returns,
    file by file, what PicketFence(path).analyze() returns -- including a file whose PixelIntensityRelationshipSign flips the values."""
    from oracle import synth
    from pylinac_b200 import picketfence as pf
    from tests.dicom_writer import write_dicom

    frames = [synth.bench_pf_frame(i) for i in range(20, 26)]
    paths = [write_dicom(tmp_path / f"pf{i}.dcm", a, pixel_spacing_mm=0.390625, sid=1000.0, gantry=0.0, coll=0.0, couch=0.0,
                         sign=-1 if i == 4 else None, slope=1.0 if i == 4 else None, intercept=0.0 if i == 4 else None)
             for i, a in enumerate(frames)]
    res = pf.analyze_files(paths, threads=4)
    assert len(res) == len(paths)
    for i in (0, 4, 5):
        single = pf.PicketFence(paths[i])
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            single.analyze()
        r = res[i]
        r.raise_for_status()
        assert int(r.s["n_meas"]) == len(single.mlc_meas) and int(r.s["n_pickets"]) == single.num_pickets
        assert float(r.s["max_error_mm"]) == pytest.approx(single.max_error, abs=1e-9)
        assert float(r.s["abs_median_error_mm"]) == pytest.approx(single.abs_median_error, abs=1e-9)


def test_picketfence_on_a_rescaled_dicom_equals_the_stored_pixels(tmp_path):
    """A clinical file with RescaleSlope / RescaleIntercept (float pixel data in the reference): the device pipeline analyses the
    stored integers (image.frame_u16); positions agree with the analysis of the raw array to fp64 rounding, counts exactly."""
    from oracle import synth
    from pylinac_b200.picketfence import PicketFence
    from tests.dicom_writer import write_dicom

    a = synth.bench_pf_frame(17)
    p = write_dicom(tmp_path / "rs.dcm", a, pixel_spacing_mm=0.390625, sid=1000.0, slope=0.37, intercept=-12.5, gantry=0.0, coll=0.0, couch=0.0)
    f1 = PicketFence(p)
    f1.analyze()
    f2 = PicketFence(a, image_kwargs={"dpi": 25.4 / 0.390625, "sid": 1000})
    f2.analyze()
    assert f1._raw.array.dtype == np.float64 and not np.array_equal(f1._raw.array, np.floor(f1._raw.array))
    assert f1.num_pickets == f2.num_pickets == 10 and len(f1.mlc_meas) == len(f2.mlc_meas) == 500
    np.testing.assert_allclose(f1._result.m["position"], f2._result.m["position"], rtol=0, atol=1e-9)
    np.testing.assert_allclose(f1.max_error, f2.max_error, rtol=0, atol=1e-9)
    # PixelIntensityRelationshipSign = -1 flips the stored values; the corner inversion check flips them back
    p3 = write_dicom(tmp_path / "neg.dcm", a, pixel_spacing_mm=0.390625, sid=1000.0, slope=1.0, intercept=0.0, sign=-1)
    f3 = PicketFence(p3)
    f3.analyze()
    assert f3.num_pickets == 10 and len(f3.mlc_meas) == 500
    np.testing.assert_allclose(np.sort(f3._result.m["position"][:, 0]), np.sort(f2._result.m["position"][:, 0]), rtol=0, atol=1e-9)
