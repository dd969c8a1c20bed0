"""CPU tests of the host-side mirror of the reference interface (no GPU): context defaults, border math, kernel taps,
the kernel-cache replay, feature objects, sharding."""
import pickle

import numpy as np
import pytest


def test_status_codes_and_defaults(golden):
    from pyfeaturetrack_b200 import klt
    s = klt.kltState
    assert (s.KLT_TRACKED, s.KLT_NOT_FOUND, s.KLT_SMALL_DET, s.KLT_MAX_ITERATIONS, s.KLT_OOB, s.KLT_LARGE_RESIDUE) == (0, -1, -2, -3, -4, -5)
    tc = klt.KLT_TrackingContext()
    assert [tc.nPyramidLevels, tc.subsampling, tc.borderx, tc.bordery] == list(golden["default_ctx"])
    assert isinstance(tc.borderx, float)                      # quirk Q1: true division
    assert (tc.mindist, tc.window_width, tc.window_height, tc.max_iterations) == (10, 7, 7, 10)
    assert tc.max_residue is None and tc.min_determinant == 0.01 and tc.min_displacement == 0.1
    assert tc.affineConsistencyCheck == -1 and tc.affine_window_width == 15
    assert tc.pyramid_last is None and not tc.sequentialMode and not tc.retainTrackers


def test_borders_and_pyramid_heuristic(golden):
    from pyfeaturetrack_b200 import klt
    for w, L, ss, border in golden["borders"]:
        tc = klt.KLT_TrackingContext()
        tc.window_width = tc.window_height = int(w)
        tc.nPyramidLevels, tc.subsampling = int(L), int(ss)
        tc.KLTUpdateTCBorder()
        assert tc.borderx == border and tc.bordery == border
    for sr, L, ss in golden["pyramid_choices"]:
        tc = klt.KLT_TrackingContext()
        tc.KLTChangeTCPyramid(int(sr))
        assert (tc.nPyramidLevels, tc.subsampling) == (int(L), int(ss))


def test_window_fixups_warn_and_mutate(capsys):
    from pyfeaturetrack_b200 import klt
    tc = klt.KLT_TrackingContext()
    tc.window_width, tc.window_height = 6, 2
    tc.KLTUpdateTCBorder()
    assert (tc.window_width, tc.window_height) == (7, 3)
    assert "must be odd" in capsys.readouterr().out


@pytest.mark.parametrize("sigma", [0.7, 1.0, 1.5, 1.8, 3.6, 7.2])
def test_kernel_taps_bit_exact(golden, sigma):
    from pyfeaturetrack_b200 import convolve
    g, d = convolve._computeKernels(sigma)
    assert np.array_equal(np.array(g), golden["taps_g_%s" % sigma])
    assert np.array_equal(np.array(d), golden["taps_d_%s" % sigma])
    assert convolve.KLTGetKernelWidths(sigma) == (len(g), len(d))
    assert convolve.cached_sigma_last == sigma


def test_kernel_too_wide_raises_nameerror_like_reference():
    from pyfeaturetrack_b200 import convolve
    with pytest.raises(NameError):
        convolve._computeKernels(14.4)


def test_kernel_cache_quirk_replayed():
    """convolve.py:236,258: a sigma within 0.05 of the cached one reuses the stale taps (quirk Q8)."""
    from pyfeaturetrack_b200 import convolve
    convolve._computeKernels(1.0)
    g_stale, _ = convolve._kernels_for_smoothing(1.04)
    assert convolve.cached_sigma_last == 1.0 and list(g_stale) == list(convolve._computeKernels(1.0)[0])
    g_new, _ = convolve._kernels_for_smoothing(1.06)
    assert convolve.cached_sigma_last == 1.06 and len(g_new) == 7


def test_taps_replay_matches_reference_cache_sequence(reference):
    """_taps_for_one_image must leave the kernel cache exactly where the reference's ComputeImagePyramids leaves it."""
    from pyfeaturetrack_b200 import klt, trackFeatures, convolve
    rklt, rconv = reference["klt"], reference["convolve"]
    for kw in (dict(), dict(nPyramidLevels=3, subsampling=2), dict(window_width=15, window_height=15),
               dict(grad_sigma=0.72), dict(nPyramidLevels=1), dict(smooth_sigma_fact=0.15, grad_sigma=1.02)):
        tc, rtc = klt.KLT_TrackingContext(), rklt.KLT_TrackingContext()
        for t in (tc, rtc):
            for k, v in kw.items():
                setattr(t, k, v)
            t.KLTUpdateTCBorder()
        taps = trackFeatures._taps_for_one_image(tc)
        # replay the reference's call sequence for one image on its own cache (trackFeatures.py:165-172)
        img = np.zeros((16, 16), np.float32)
        rconv.KLTComputeSmoothedImage(img, rtc.smooth_sigma_fact * max(rtc.window_width, rtc.window_height))
        smooth_ref = list(rconv.cachegauss)
        for _ in range(1, rtc.nPyramidLevels):
            rconv.KLTComputeSmoothedImage(img, rtc.subsampling * rtc.pyramid_sigma_fact)
        pyr_ref = list(rconv.cachegauss)
        for _ in range(rtc.nPyramidLevels):
            rconv.KLTComputeGradients(img, rtc.grad_sigma)
        assert list(taps.smooth.taps[:taps.smooth.n]) == smooth_ref
        if rtc.nPyramidLevels > 1:
            assert list(taps.pyramid.taps[:taps.pyramid.n]) == pyr_ref
        assert list(taps.grad_gauss.taps[:taps.grad_gauss.n]) == list(rconv.cachegauss)
        assert list(taps.grad_deriv.taps[:taps.grad_deriv.n]) == list(rconv.cachegaussderiv)
        assert convolve.cached_sigma_last == rconv.cached_sigma_last


def test_feature_objects():
    from pyfeaturetrack_b200 import klt
    f = klt.KLT_Feature()
    assert not hasattr(f, "x") and not hasattr(f, "val")      # quirk Q5
    f.x, f.y, f.val = 1.5, 2.5, 0
    g = pickle.loads(pickle.dumps([f]))[0]
    assert (g.x, g.y, g.val) == (1.5, 2.5, 0)
    h = klt.KLT_Feature(); h.x = h.y = -1.0; h.val = -4
    assert klt.KLTCountRemainingFeatures([f, h]) == 1


def test_params_struct_from_context():
    from pyfeaturetrack_b200 import klt, selectGoodFeatures as sgf
    tc = klt.KLT_TrackingContext()
    p = sgf.make_params(tc)
    assert (p.window_width, p.n_levels, p.subsampling, p.has_max_residue) == (7, 2, 4, 0)
    assert p.borderx == 30.0
    tc.max_residue = 10.0
    tc.retainTrackers = True
    p = sgf.make_params(tc)
    assert p.has_max_residue == 1 and p.max_residue == 10.0 and p.retain_trackers == 1


def test_unported_paths_fail_like_the_reference(img01):
    from pyfeaturetrack_b200 import klt, trackFeatures as tf
    tf.KLT_verbose = 0
    tc = klt.KLT_TrackingContext()
    f = klt.KLT_Feature(); f.x, f.y, f.val = 100.0, 100.0, 0
    tc.lighting_insensitive = True
    tc.affineConsistencyCheck = 2      # lighting_insensitive alone is implemented here (the reference raises); with affine it is not
    with pytest.raises(Exception, match="Not implemented"):
        tf.KLTTrackFeatures(tc, img01[0], img01[1], [f])
    with pytest.raises(AssertionError):
        tf.KLTTrackFeatures(klt.KLT_TrackingContext(), img01[0], img01[1][:100], [f])


def test_install_dropin_aliases_reference_module_names():
    import sys
    import pyfeaturetrack_b200 as P
    saved = {k: sys.modules.get(k) for k in P.DROPIN_MODULES}
    try:
        P.install_dropin()
        import klt, selectGoodFeatures, trackFeatures, convolve, pyramid, goodFeaturesUtils, trackFeaturesUtils  # noqa
        assert klt.KLT_TrackingContext is P.klt.KLT_TrackingContext
        assert hasattr(selectGoodFeatures, "KLTSelectGoodFeatures") and hasattr(trackFeatures, "KLTTrackFeatures")
        assert hasattr(goodFeaturesUtils, "ScanImageForGoodFeatures") and hasattr(trackFeaturesUtils, "extractImagePatchSlow")
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_shard_range_partitions():
    from pyfeaturetrack_b200.shard import shard_range
    for n in (0, 1, 7, 8, 300, 2401):
        for world in (1, 2, 3, 8):
            got = [u for r in range(world) for u in shard_range(n, r, world)]
            assert got == list(range(n))
            sizes = [len(shard_range(n, r, world)) for r in range(world)]
            assert max(sizes) - min(sizes) <= 1


def test_write_feature_list_roundtrip(tmp_path, img01):
    """C-KLT 1.3.4's feature-list files (the format the reference's stubs at writeFeatures.py:53-82 name the helpers of):
    text with "%5.1f" and "%3d", binary "KLTFL1", and both read back."""
    from pyfeaturetrack_b200 import klt, writeFeatures as wf, selectGoodFeatures as sgf
    sgf.KLT_verbose = 0
    fl = []
    for i in range(5):
        f = klt.KLT_Feature(); f.x, f.y, f.val = 10.5 + i, 20.25 + 2 * i, (11046 if i % 2 == 0 else -4)
        if i % 2:
            f.x = f.y = -1.0
        fl.append(f)
    wf.KLTWriteFeatureList(fl, str(tmp_path / "fl.bin"), None)
    raw = open(str(tmp_path / "fl.bin"), "rb").read()
    assert raw[:6] == b"KLTFL1" and len(raw) == 6 + 4 + 5 * 12
    back = wf.KLTReadFeatureList(str(tmp_path / "fl.bin"))
    assert [(f.x, f.y, f.val) for f in back] == [(f.x, f.y, f.val) for f in fl]
    wf.KLTWriteFeatureList(fl, str(tmp_path / "fl.txt"), "%5.1f")
    text = open(str(tmp_path / "fl.txt")).read()
    assert text.startswith("Feel free to place comments here.\n\n\n\n!!! Warning:  This is a KLT data file.  ")
    assert "------------------------------\nKLT Feature List\n------------------------------\n\nnFeatures = 5\n\n" in text
    assert "feature | (x,y)=val\n--------+-" + "-" * 20 + "\n" in text
    assert "      0 | ( 10.5, 20.2)=11046 \n" in text
    assert "      1 | ( -1.0, -1.0)=   -4 \n" in text
    back = wf.KLTReadFeatureList(str(tmp_path / "fl.txt"))
    assert [(f.x, f.val) for f in back] == [(10.5, 11046), (-1.0, -4), (12.5, 11046), (-1.0, -4), (14.5, 11046)]
    wf.KLTWriteFeatureList(fl, str(tmp_path / "fl3.txt"), "%3d")
    text = open(str(tmp_path / "fl3.txt")).read()
    assert "      0 | ( 11, 20)=11046 \n" in text and "      1 | ( -1, -1)=   -4 \n" in text     # rounded unless negative
    assert "--------+-" + "-" * 16 + "\n" in text
    with pytest.raises(ValueError):
        wf.KLTWriteFeatureList(fl, str(tmp_path / "bad.txt"), "5.1f")
    wf.KLTWriteFeatureListToPPM(fl, img01[0], str(tmp_path / "f.ppm"))
    from PIL import Image
    rgb = np.array(Image.open(str(tmp_path / "f.ppm")))
    assert tuple(rgb[20, 11]) == (255, 0, 0) and tuple(rgb[22, 12]) != (255, 0, 0)     # feature 0 drawn, feature 1 (lost) not


def test_ppm_overlay_equals_the_reference_file(tmp_path, img01, reference):
    """KLTWriteFeatureListToPPM against the reference's own function (writeFeatures.py:10-37): same bytes, including features
    on the image border, rounded positions and lost features."""
    if "writeFeatures" not in reference:
        pytest.skip("oracle/_ref predates writeFeatures (python oracle/build_ref.py --force)")
    from PIL import Image
    from pyfeaturetrack_b200 import klt, writeFeatures as wf, selectGoodFeatures as sgf
    sgf.KLT_verbose = 0
    img = Image.fromarray(img01[0]) if isinstance(img01[0], np.ndarray) else img01[0]
    w, h = img.size
    rng = np.random.default_rng(2)
    fl = []
    for i in range(60):
        f = klt.KLT_Feature()
        f.x, f.y = float(rng.uniform(0, w - 1)), float(rng.uniform(0, h - 1))
        f.val = int(rng.integers(-5, 5000))
        fl.append(f)
    for x, y in ((0.0, 0.0), (w - 1.0, h - 1.0), (0.4, h - 1.4), (w - 0.6, 0.49)):      # corners and edges
        f = klt.KLT_Feature(); f.x, f.y, f.val = x, y, 7
        fl.append(f)
    ours, theirs = str(tmp_path / "ours.ppm"), str(tmp_path / "theirs.ppm")
    wf.KLTWriteFeatureListToPPM(fl, img, ours)
    reference["writeFeatures"].KLTWriteFeatureListToPPM(fl, img, theirs)
    assert open(ours, "rb").read() == open(theirs, "rb").read()


def test_precision_modes_and_host_binding():
    """config: 'windowed' is a tracking-only mode; the NUMA binding helper is a no-op without NVML/GPU."""
    import pytest
    from pyfeaturetrack_b200 import config, _capi, shard
    saved = (config.track_precision, config.select_precision, config.operator_precision)
    try:
        config.set_precision(track="windowed")
        assert config.track_precision_code() == _capi.PRECISION_FAST_WINDOWED == 2
        config.set_precision(track="fast", select="strict", operator="fast")
        assert (config.track_precision_code(), config.select_precision_code(), config.operator_precision_code()) == (0, 1, 0)
        config.set_precision(track="auto")
        px = 1920 * 1080
        assert config.track_precision_code() == 2 and config.track_precision_code(1000, px) == 2      # sparse: windowed
        assert config.track_precision_code(px // config.AUTO_PIXELS_PER_FEATURE + 1, px) == 0          # dense: planes
        for bad in (dict(select="windowed"), dict(operator="auto"), dict(track="exact")):
            with pytest.raises(ValueError):
                config.set_precision(**bad)
    finally:
        config.set_precision(track=saved[0], select=saved[1], operator=saved[2])
    import torch
    if not torch.cuda.is_available():
        assert shard.bind_host_to_gpu(0) == 0


def test_oracle_lighting_insensitive_restatement():
    """Lighting-insensitive tracking, restated from the C the reference carries as comments (trackFeaturesUtils.pyx:152-239;
    the reference raises instead): under a gain + bias change of the second frame the plain tracker rejects most features
    with KLT_LARGE_RESIDUE, the normalised one keeps tracking them to the same displacement."""
    from oracle import klt_oracle as O
    from pyfeaturetrack_b200 import synth
    a, b = synth.frame_pair(240, 320, seed=5, shift=(1.6, -2.2))
    dim = np.clip(0.6 * b.astype(np.float32) + 40, 0, 255).astype(np.uint8)
    res = {}
    for li in (False, True):
        p = O.Params(nPyramidLevels=2, subsampling=2, max_residue=10.0, lighting_insensitive=li)
        sel = O.select_good_features(p, a, 100)
        for name, img2 in (("same", b), ("dim", dim)):
            x, y, v, _ = O.track_features(p, a, img2, *sel)
            ok = v == 0
            res[(li, name)] = (int(ok.sum()), float(np.median((x - sel[0])[ok])), float(np.median((y - sel[1])[ok])), v)
    assert res[(False, "same")][0] >= 90 and res[(True, "same")][0] >= 90
    assert res[(False, "dim")][0] < 40 and (res[(False, "dim")][3] == -5).sum() > 50     # large residue without normalisation
    assert res[(True, "dim")][0] >= 80                                                  # recovered with it
    for k in ((True, "same"), (True, "dim")):
        assert abs(res[k][1] - res[(False, "same")][1]) < 0.1 and abs(res[k][2] - res[(False, "same")][2]) < 0.1


def test_feature_table_and_history_round_trip():
    """storeFeatures: the table/history routines the reference only declares (klt.py:272-283)."""
    from pyfeaturetrack_b200 import storeFeatures as sf, klt
    nframes, nfeat = 4, 5
    ft = sf.KLTCreateFeatureTable(nframes, nfeat)
    fl = sf.KLTCreateFeatureList(nfeat)
    for frame in range(nframes):
        for i, f in enumerate(fl):
            f.x, f.y, f.val = 10.0 * i + frame, 2.0 * i - frame, (0 if frame else 100 + i) if i != 3 or frame < 2 else -4
        sf.KLTStoreFeatureList(fl, ft, frame)
    out = sf.KLTCreateFeatureList(nfeat)
    sf.KLTExtractFeatureList(out, ft, 2)
    assert [(f.x, f.y, f.val) for f in out] == [(10.0 * i + 2, 2.0 * i - 2, 0 if i != 3 else -4) for i in range(nfeat)]
    fh = sf.KLTCreateFeatureHistory(nframes)
    sf.KLTExtractFeatureHistory(fh, ft, 3)
    assert [r.val for r in fh.feature] == [103, 0, -4, -4]
    fh.feature[1].x = 999.0
    sf.KLTStoreFeatureHistory(fh, ft, 3)
    x, y, v = sf.table_arrays(ft)
    assert x.shape == (nfeat, nframes) and x[3, 1] == 999.0 and v[3, 3] == -4 and v[0, 0] == 100
    with pytest.raises(SystemExit):
        sf.KLTStoreFeatureList(fl, ft, nframes)                   # frame out of range: KLTError exits like the C library
    with pytest.raises(SystemExit):
        sf.KLTStoreFeatureList(fl[:-1], ft, 0)
    assert isinstance(ft, klt.KLT_FeatureTable) and isinstance(fh, klt.KLT_FeatureHistory)


def test_featlist_helper_matches_python_walks():
    """csrc/featlist.c (the list <-> arrays walks of KLTTrackFeatures through the CPython C API) against the Python loops it
    replaces: mixed Python / NumPy scalar attributes, lost features, affine templates dropped with the feature."""
    import copy
    from pyfeaturetrack_b200 import _capi, build, klt, trackFeatures as tf
    build.build_featlist()
    _capi._featlist = False
    L = _capi.featlist()
    assert L is not None
    rng = np.random.default_rng(5)
    fl = []
    for i in range(257):
        f = klt.KLT_Feature()
        f.x = np.int32(i) if i % 3 else float(i) + 0.25
        f.y = float(rng.uniform(0, 500))
        f.val = int(rng.integers(-5, 3)) if i % 2 else np.int32(rng.integers(-5, 3))
        if i % 4 == 0:
            f.aff_img, f.aff_img_gradx, f.aff_img_grady = "t", "gx", "gy"
        fl.append(f)
    x, y, val = tf._features_to_arrays(fl)
    _capi._featlist = None
    try:
        x2, y2, val2 = tf._features_to_arrays(fl)
    finally:
        _capi._featlist = False
    assert np.array_equal(x, x2) and np.array_equal(y, y2) and np.array_equal(val, val2)
    assert val.dtype == np.int32 and np.all(x[val < 0] == -1.0)
    new_val = rng.integers(-4, 1, len(fl)).astype(np.int32)
    nx, ny = x + 0.5, y - 0.25
    a, b = copy.deepcopy(fl), copy.deepcopy(fl)
    L.klt_featlist_scatter_tracked(a, len(a), nx.ctypes.data, ny.ctypes.data, new_val.ctypes.data, val.ctypes.data)
    for feat, live, fx, fy, v in zip(b, (val >= 0).tolist(), nx.tolist(), ny.tolist(), new_val.tolist()):
        if not live:
            continue
        if v == 0:
            feat.x, feat.y, feat.val = fx, fy, 0
        else:
            feat.x, feat.y, feat.val = -1.0, -1.0, v
            if "aff_img" in feat.__dict__:
                tf._clear_affine(feat)
    for fa, fb in zip(a, b):
        assert fa.__dict__ == fb.__dict__
        assert type(fa.val) is type(fb.val) and type(fa.x) is type(fb.x)
    with pytest.raises(AttributeError):
        L.klt_featlist_gather([1, 2], 2, x.ctypes.data, y.ctypes.data, val.ctypes.data)


def test_pil_pixels_into_staging_array():
    """_pil_into: PIL 'L' image -> uint8 array in one pass (core paste) and through the chunked raw encoder, odd sizes included."""
    from PIL import Image
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf
    rng = np.random.default_rng(11)
    for shape in ((37, 53), (240, 320), (481, 643), (1080, 1920)):
        a = rng.integers(0, 256, shape, dtype=np.uint8)
        img = Image.fromarray(a)
        stage = np.zeros(shape, np.uint8)
        sgf._pil_into(stage, img, shape[1], shape[0])
        assert np.array_equal(stage, a)
        # the encoder path (what runs if frombuffer / core paste are not available)
        real = Image.frombuffer
        try:
            Image.frombuffer = None
            sgf._pil_views.clear()
            stage[:] = 0
            sgf._pil_into(stage, img, shape[1], shape[0])
        finally:
            Image.frombuffer = real
            sgf._pil_views.clear()
        assert np.array_equal(stage, a)


def test_bench_has_no_collective_after_the_ranks_leave():
    """bench.py at N > 1: ranks != 0 destroy their process group and return once the timed sections are over; anything rank 0
    runs after that point must be local.  (A barrier there hangs the N > 1 run until the launcher's timeout.)"""
    import ast
    import os
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")).read()
    fn = [n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == "run_b200"][0]
    leave = [i for i, st in enumerate(fn.body) if isinstance(st, ast.If) and ast.unparse(st.test) == "rank != 0"]
    assert len(leave) == 1
    collective = {"timed", "barrier", "run_e2e", "run_e2e_async", "sequence_bench", "all_reduce", "all_gather", "broadcast",
                  "gather_features", "init_process_group"}
    for st in fn.body[leave[0] + 1:]:
        for node in ast.walk(st):
            if isinstance(node, ast.Call):
                name = node.func.attr if isinstance(node.func, ast.Attribute) else getattr(node.func, "id", "")
                assert name not in collective, "collective call %s() after ranks != 0 have left (line %d)" % (name, node.lineno)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the reference's own CPU path from oracle/_ref, no GPU): one JSON line with the contract's keys,
    the metric / unit / config of the B200 arm, e2e == value with zero copies, and a cpu_baseline that describes the run."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if not os.path.isdir(os.path.join(root, "oracle", "_ref")):
        pytest.skip("oracle/_ref not built")
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--ref-procs", "2"], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "tracked_features_per_sec" and d["unit"] == "tracked features/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] == 2 and d["cpu_baseline"]["value"] == d["value"]
    sys.path.insert(0, root)
    import bench
    assert d["config"] == bench.bench_config(bench.WORKLOADS["B"])      # the B200 arm prints the same object


def test_bench_select_fast_leg_on_stubs(monkeypatch):
    """bench.py's `select_fast` leg (north_star (2): fused fast selection, batched) against a stubbed GPU library: the Python
    of the leg runs, and its byte accounting is what DESIGN states (4 B/px read + 4 B/candidate written for the fused pass)."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import _bench_flow_driver as drv
    import bench
    from pyfeaturetrack_b200 import _capi, klt, selectGoodFeatures as sgf, trackFeatures as tf

    class Ctx(drv.FakeCtx):
        def profile_read(self):
            return {"eigen_fast": dict(ms=0.3, launches=3, bytes=0.0), "select_walk": dict(ms=0.15, launches=3, bytes=0.0)}

    monkeypatch.setattr(_capi, "Pyramid", drv.FakePyramid)
    wl = dict(bench.WORKLOADS["B"], H=48, W=64, n=10)
    distinct = [(np.zeros((48, 64), np.uint8), np.zeros((48, 64), np.uint8))]
    r = bench.select_fast_timing(Ctx(), drv.FakeLib(), _capi, klt, sgf, tf, distinct, wl, 6553.0, batch=4, reps=2)
    assert r["ms_per_call"] == 0.5 and r["ms_per_frame"] == 0.125 and r["kernel_ms_per_call"]["eigen_fast"] == 0.1
    fused, unfused = r["eigen_pass"]["bytes_per_frame_fused"], r["eigen_pass"]["bytes_per_frame_unfused_accounting"]
    assert fused >= 4.0 * 64 * 48 and (fused - 4.0 * 64 * 48) % 4 == 0 and unfused - fused == 13.0 * 64 * 48


def test_bench_dump_outputs(tmp_path, monkeypatch):
    """bench.py --dump-outputs: the timed step's x / y / val lists as float64 .npy files, the same seeded sample of pairs on every
    run once the lists exceed the size limit, and per-rank names at N > 1.  The device arrays are stood in by host arrays."""
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench

    class Ctx(object):
        def memcpy(self, dst, src, nbytes):
            assert dst.nbytes == nbytes == src.nbytes
            dst[...] = src

        def sync(self):
            pass

    B, n = 12, 5
    rng = np.random.default_rng(1)
    x, y = rng.uniform(0, 100, (B, n)), rng.uniform(0, 100, (B, n))
    v = rng.integers(-5, 1, (B, n)).astype(np.int32)
    bench.dump_outputs(str(tmp_path / "all"), Ctx(), x, y, v, B, n, 0, 1)
    got = {k: np.load(str(tmp_path / "all" / (k + ".npy"))) for k in ("x", "y", "val")}
    assert sorted(os.listdir(str(tmp_path / "all"))) == ["val.npy", "x.npy", "y.npy"]
    assert all(a.dtype == np.float64 and a.shape == (B, n) for a in got.values())
    assert np.array_equal(got["x"], x) and np.array_equal(got["y"], y) and np.array_equal(got["val"], v)

    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 5 * (3 * n + 1) * 8)       # room for 5 pairs
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), Ctx(), x, y, v, B, n, 0, 1)
    pairs = np.load(str(tmp_path / "s1" / "pairs.npy"))
    assert np.array_equal(pairs, np.load(str(tmp_path / "s2" / "pairs.npy")))
    assert len(pairs) == 5 and np.all(np.diff(pairs) > 0)
    pick = pairs.astype(np.int64)
    assert np.array_equal(np.load(str(tmp_path / "s1" / "x.npy")), x[pick])
    assert np.array_equal(np.load(str(tmp_path / "s1" / "val.npy")), v[pick])
    assert sum(os.path.getsize(str(tmp_path / "s1" / f)) - 128 for f in os.listdir(str(tmp_path / "s1"))) <= bench.DUMP_LIMIT_BYTES

    bench.dump_outputs(str(tmp_path / "r"), Ctx(), x, y, v, B, n, 1, 2)
    assert sorted(os.listdir(str(tmp_path / "r"))) == ["pairs_rank1.npy", "val_rank1.npy", "x_rank1.npy", "y_rank1.npy"]
