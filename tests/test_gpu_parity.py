"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI (ctypes shims in
pyfeaturetrack_b200), against the CPU oracle on the same seeded inputs and against the reference's golden vectors.

Bars (BASELINE.json north_star): STRICT mode is bit-exact everywhere (images, eigen map, selection, positions, status
codes).  FAST mode: images within 1e-5 relative-to-max, positions within 1e-3 px, status codes >= 99.9 %."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REL_TOL = 1e-5        # images, relative to the image's max |value|
POS_TOL = 1e-3        # px
STATUS_MATCH = 0.999


def P(oracle, **kw):
    return oracle.Params(**kw)


def fl(golden, key):
    a = golden[key]
    return a[0], a[1], a[2].astype(np.int32)


def make_tc(**kw):
    from pyfeaturetrack_b200 import klt
    tc = klt.KLT_TrackingContext()
    for k, v in kw.items():
        setattr(tc, k, v)
    tc.KLTUpdateTCBorder()
    return tc


def fl_arrays(featurelist):
    return (np.array([float(f.x) for f in featurelist]), np.array([float(f.y) for f in featurelist]),
            np.array([int(f.val) for f in featurelist], np.int32))


def assert_features_equal(got, want):
    assert np.array_equal(np.asarray(got[2], np.int64), np.asarray(want[2], np.int64))
    assert np.array_equal(np.asarray(got[0], np.float64), np.asarray(want[0], np.float64))
    assert np.array_equal(np.asarray(got[1], np.float64), np.asarray(want[1], np.float64))


def assert_features_close(got, want):
    gv, wv = np.asarray(got[2]), np.asarray(want[2])
    match = np.mean(gv == wv)
    assert match >= STATUS_MATCH, "status match %.4f" % match
    both = (gv == 0) & (wv == 0)
    err = np.maximum(np.abs(np.asarray(got[0])[both] - np.asarray(want[0])[both]),
                     np.abs(np.asarray(got[1])[both] - np.asarray(want[1])[both]))
    assert err.size == 0 or err.max() <= POS_TOL, "max position error %g px" % err.max()


@pytest.fixture(autouse=True)
def _quiet():
    from pyfeaturetrack_b200 import selectGoodFeatures, trackFeatures, config
    selectGoodFeatures.KLT_verbose = 0
    trackFeatures.KLT_verbose = 0
    config.set_precision(track="fast", select="strict", operator="strict")
    yield


# ---- convolution operators -------------------------------------------------------------------------------------
@pytest.mark.parametrize("sigma", [0.7, 1.0, 1.5, 1.8, 3.6, 7.2])
@pytest.mark.parametrize("shape", [(77, 123), (240, 320), (33, 40)])
def test_smooth_and_gradients(gpu_ctx, oracle, sigma, shape):
    from pyfeaturetrack_b200 import convolve, config
    rng = np.random.default_rng(int(sigma * 10) + shape[0])
    img = (rng.random(shape) * 255).astype(np.float32)
    cache = oracle.KernelCache()
    want_s = oracle.smooth(img, sigma, cache)
    want_gx, want_gy = oracle.gradients(img, sigma, cache)
    convolve._computeKernels(sigma)
    config.set_precision(operator="strict")
    assert np.array_equal(convolve.KLTComputeSmoothedImage(img, sigma), want_s)
    gx, gy = convolve.KLTComputeGradients(img, sigma)
    assert np.array_equal(gx, want_gx) and np.array_equal(gy, want_gy)
    config.set_precision(operator="fast")
    s = convolve.KLTComputeSmoothedImage(img, sigma)
    gx, gy = convolve.KLTComputeGradients(img, sigma)
    assert np.abs(s - want_s).max() <= REL_TOL * np.abs(want_s).max()
    assert np.abs(gx - want_gx).max() <= REL_TOL * max(np.abs(want_gx).max(), np.abs(want_s).max())
    assert np.abs(gy - want_gy).max() <= REL_TOL * max(np.abs(want_gy).max(), np.abs(want_s).max())


def test_golden_images(gpu_ctx, golden, img01):
    from pyfeaturetrack_b200 import convolve, pyramid
    convolve._computeKernels(0.7)
    sm = convolve.KLTComputeSmoothedImage(img01[0].astype(np.float32), 0.7)
    assert np.array_equal(sm, golden["A_smooth"])
    convolve._computeKernels(1.0)
    gx, gy = convolve.KLTComputeGradients(sm, 1.0)
    assert np.array_equal(gx, golden["A_gradx"]) and np.array_equal(gy, golden["A_grady"])
    p = pyramid.KLTPyramid(320, 240, 4, 2)
    p.Compute(sm, 0.9)
    assert p.img[0] is sm
    assert np.array_equal(p.img[1], golden["A_pyr1"])
    assert p.ncols == [320, 80.0] and p.nrows == [240, 60.0]


def test_general_kernel_and_wide_kernel(gpu_ctx, oracle):
    """Non-symmetric taps take SciPy's general branch; a kernel wider than the image exercises repeated reflection."""
    from pyfeaturetrack_b200 import convolve
    rng = np.random.default_rng(3)
    img = (rng.random((20, 31)) * 100).astype(np.float32)
    hk = rng.random(7)
    vk = rng.random(5)
    assert np.array_equal(convolve._convolveSeparate(img, hk, vk), oracle.conv_separable(img, hk, vk))
    g, d = oracle.compute_kernels(7.2)       # 43 / 51 taps on a 20-row image
    assert np.array_equal(convolve._convolveSeparate(img, d, g), oracle.conv_separable(img, d, g))


# ---- pyramids ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [dict(shape=(240, 320), L=2, ss=4), dict(shape=(480, 640), L=3, ss=2),
                                 dict(shape=(270, 350), L=2, ss=8), dict(shape=(203, 301), L=3, ss=2),
                                 dict(shape=(120, 160), L=1, ss=2)])
def test_pyramid_build_u8(gpu_ctx, oracle, cfg):
    from pyfeaturetrack_b200 import _capi, trackFeatures
    rng = np.random.default_rng(cfg["L"] * 7 + cfg["ss"])
    H, W = cfg["shape"]
    batch = 3
    frames = (rng.random((batch, H, W)) * 255).astype(np.uint8)
    p = P(oracle, nPyramidLevels=cfg["L"], subsampling=cfg["ss"])
    tc = make_tc(nPyramidLevels=cfg["L"], subsampling=cfg["ss"])
    pyr = _capi.Pyramid(gpu_ctx, W, H, cfg["L"], cfg["ss"], batch)
    for prec in (_capi.PRECISION_STRICT, _capi.PRECISION_FAST):
        pyr.build_u8(frames, trackFeatures._taps_for_one_image(tc), prec)
        for b in range(batch):
            want = oracle.image_pyramids(p, frames[b])
            for which in range(3):
                for lvl in range(cfg["L"]):
                    got = pyr.download(which, lvl, b)
                    ref = want[which][lvl]
                    assert got.shape == ref.shape
                    if prec == _capi.PRECISION_STRICT:
                        assert np.array_equal(got, ref), (b, which, lvl)
                    else:
                        assert np.abs(got - ref).max() <= REL_TOL * 255.0, (b, which, lvl)
    pyr.close()


@pytest.mark.parametrize("cfg", [dict(shape=(1080, 1920), L=3, batch=3), dict(shape=(200, 360), L=2, batch=2),
                                 dict(shape=(64, 248), L=2, batch=1), dict(shape=(540, 964), L=3, batch=2),
                                 dict(shape=(2160, 3840), L=4, batch=1), dict(shape=(97, 132), L=2, batch=4),
                                 dict(shape=(72, 116), L=2, batch=2)])
def test_image_only_pyramids_vs_oracle(gpu_ctx, oracle, cfg):
    """The image-only (windowed) build -- the packed two-strip level-0 kernel and the packed decimation -- against the
    oracle's pyramids: odd and even strip counts, a strip pair whose second strip lies outside the image, a single strip,
    segments that touch the top / bottom border and interior ones, widths that are not multiples of 120."""
    from pyfeaturetrack_b200 import _capi, trackFeatures
    H, W = cfg["shape"]
    L, batch = cfg["L"], cfg["batch"]
    frames = (np.random.default_rng(H * 3 + W).random((batch, H, W)) * 255).astype(np.uint8)
    p = P(oracle, nPyramidLevels=L, subsampling=2)
    tc = make_tc(nPyramidLevels=L, subsampling=2)
    pyr = _capi.Pyramid(gpu_ctx, W, H, L, 2, batch)
    pyr.build_u8(frames, trackFeatures._taps_for_one_image(tc), _capi.PRECISION_FAST_WINDOWED)
    for b in range(batch):
        want = oracle.image_pyramids(p, frames[b])
        for lvl in range(L):
            got = pyr.download(0, lvl, b)
            assert got.shape == want[0][lvl].shape
            assert np.abs(got - want[0][lvl]).max() <= REL_TOL * 255.0, (b, lvl)
    pyr.close()


def test_kernel_generations_agree(gpu_ctx):
    """The image-only (windowed) build starts with the fused level-0 + level-1 kernel (stream_level01) where it can, and
    otherwise with the level-0 kernel (stream_smooth0x2) followed by the packed decimation (stream_down2).  The fused
    kernel needs a frame pitch that is a multiple of 8, so the same frames, once contiguous and once in a buffer with 4
    bytes of padding per row, take the two paths.  Both smooth level 0 with the same operations in the same order: level
    0 is bit-identical.  The fused kernel decimates the smoothed reflect-extended frame instead of the reflect-extended
    smoothed image: levels >= 1 agree to rounding."""
    from pyfeaturetrack_b200 import _capi, trackFeatures
    for (H, W, L, batch) in [(1080, 1920, 3, 5), (200, 360, 2, 2), (64, 248, 2, 1)]:
        frames = (np.random.default_rng(H + W).random((batch, H, W)) * 255).astype(np.uint8)
        padded = np.zeros((batch, H, W + 4), np.uint8)
        padded[:, :, :W] = frames
        taps = trackFeatures._taps_for_one_image(make_tc(nPyramidLevels=L, subsampling=2))
        levels = []
        for buf, first_kernel in ((frames, "stream_level01"), (padded, "stream_smooth0")):
            pyr = _capi.Pyramid(gpu_ctx, W, H, L, 2, batch)
            gpu_ctx.profile(True)
            gpu_ctx.profile_reset()
            try:
                pyr.build_u8(buf, taps, _capi.PRECISION_FAST_WINDOWED)      # pitch: the buffer's row length
                assert first_kernel in gpu_ctx.profile_read(), (H, W)
            finally:
                gpu_ctx.profile(False)
            levels.append([[pyr.download(0, lvl, b) for lvl in range(L)] for b in range(batch)])
            pyr.close()
        for b in range(batch):
            assert np.array_equal(levels[0][b][0], levels[1][b][0]), (H, W, b)
            for lvl in range(1, L):
                fused, split = levels[0][b][lvl], levels[1][b][lvl]
                s1, s2 = fused.sum(dtype=np.float64), split.sum(dtype=np.float64)
                assert abs(s1 - s2) <= 1e-6 * max(abs(s1), 1.0), (H, W, b, lvl)
                assert np.abs(fused - split).max() <= 1e-5 * 255.0, (H, W, b, lvl)


# ---- selection -----------------------------------------------------------------------------------------------------
def test_scan_bit_exact(gpu_ctx, oracle, golden):
    from pyfeaturetrack_b200 import goodFeaturesUtils
    px, py, pv = goodFeaturesUtils.ScanImageForGoodFeatures(golden["A_gradx"], golden["A_grady"], 30.0, 30.0, 3.5, 3.5, 0)
    assert np.array_equal(np.array(pv, np.float32).reshape(180, 260), golden["A_scan_val"])
    assert list(px[:5]) == list(golden["A_scan_x0"]) and list(py[:5]) == list(golden["A_scan_y0"])
    assert isinstance(px[0], np.int32) and isinstance(pv[0], float)
    rng = np.random.default_rng(1)
    gx = (rng.standard_normal((150, 211)) * 20).astype(np.float32)
    gy = (rng.standard_normal((150, 211)) * 20).astype(np.float32)
    for (b, hw, skip) in ((8, 3, 0), (12, 7, 1), (9, 2, 3)):
        xs, ys, val = goodFeaturesUtils.scan_values(gx, gy, b, b, hw, hw, skip)
        want, wxs, wys = oracle.scan_good_features(gx, gy, b, b, hw, hw, skip)
        assert np.array_equal(xs, wxs) and np.array_equal(ys, wys) and np.array_equal(val, want)
    with pytest.raises(ValueError):
        goodFeaturesUtils.ScanImageForGoodFeatures(gx.astype(np.float64), gy, 8, 8, 3, 3, 0)


@pytest.mark.parametrize("n", [50, 100])
def test_config_A_dropin_api(gpu_ctx, golden, img01, n):
    """example1.py's flow through the drop-in modules, PIL images in, feature list out."""
    from PIL import Image
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    config.set_precision(track="strict")
    tc = make_tc(max_residue=10.0)
    i0, i1 = Image.fromarray(img01[0]), Image.fromarray(img01[1])
    featurelist = sgf.KLTSelectGoodFeatures(tc, i0, n)
    assert_features_equal(fl_arrays(featurelist), fl(golden, "A_sel%d" % n))
    assert isinstance(featurelist[0].x, np.int32) and isinstance(featurelist[0].val, int)
    assert featurelist[0].aff_Axx == 1.0 and featurelist[0].aff_img is None
    assert tf.KLTTrackFeatures(tc, i0, i1, featurelist) is None
    assert_features_equal(fl_arrays(featurelist), fl(golden, "A_trk%d" % n))
    assert isinstance(featurelist[0].x, float)
    tf.KLTTrackFeatures(tc, i1, i0, featurelist)
    assert_features_equal(fl_arrays(featurelist), fl(golden, "A_trk%d_back" % n))
    # fast pyramids: tolerance instead of bit equality
    config.set_precision(track="fast")
    featurelist = sgf.KLTSelectGoodFeatures(tc, i0, n)
    tf.KLTTrackFeatures(tc, i0, i1, featurelist)
    assert_features_close(fl_arrays(featurelist), fl(golden, "A_trk%d" % n))


def test_selection_variants(gpu_ctx, golden, img01):
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf
    tc = make_tc(nSkippedPixels=2, mindist=15, min_eigenvalue=500)
    assert_features_equal(fl_arrays(sgf.KLTSelectGoodFeatures(tc, img01[0], 40)), fl(golden, "A_sel40_skip2"))
    tc = make_tc(smoothBeforeSelecting=False)
    assert_features_equal(fl_arrays(sgf.KLTSelectGoodFeatures(tc, img01[0], 40)), fl(golden, "A_sel40_nosmooth"))
    # flat image: candidates run out (quirk Q6) -> C-KLT fill
    tc = make_tc()
    fl_ = sgf.KLTSelectGoodFeatures(tc, np.full((120, 160), 77, np.uint8), 10)
    assert all(f.val == -1 and f.x == -1 and f.y == -1 for f in fl_)


def test_tracking_variants_strict(gpu_ctx, golden, img01):
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    config.set_precision(track="strict")
    tc = make_tc()
    f = sgf.KLTSelectGoodFeatures(tc, img01[0], 60)
    tf.KLTTrackFeatures(tc, img01[0], img01[1], f)
    assert_features_equal(fl_arrays(f), fl(golden, "A_trk60_nores"))
    tc = make_tc(retainTrackers=True)
    f = sgf.KLTSelectGoodFeatures(tc, img01[0], 60)
    tf.KLTTrackFeatures(tc, img01[0], img01[1], f)
    assert_features_equal(fl_arrays(f), fl(golden, "A_trk60_retain"))


def test_sequential_mode_with_replacement(gpu_ctx, golden, img01):
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    config.set_precision(track="strict")
    tc = make_tc(max_residue=10.0, sequentialMode=True)
    f = sgf.KLTSelectGoodFeatures(tc, img01[0], 80)
    want = golden["A_seq80"]
    k = 0
    for a, b in ((0, 1), (1, 0), (0, 1)):
        tf.KLTTrackFeatures(tc, img01[a], img01[b], f)
        assert_features_equal(fl_arrays(f), (want[k][0], want[k][1], want[k][2]))
        k += 1
        sgf.KLTReplaceLostFeatures(tc, img01[b], f)
        assert_features_equal(fl_arrays(f), (want[k][0], want[k][1], want[k][2]))
        k += 1
    assert tc.pyramid_last.img[0].shape == (240, 320)      # NumPy view of the device pyramid on demand
    import pickle
    pickle.loads(pickle.dumps(f))
    pickle.loads(pickle.dumps(tc))


def _synth(seed, shape=(480, 640), shift=(1.7, -3.3)):
    from pyfeaturetrack_b200 import synth
    return synth.frame_pair(shape[0], shape[1], seed=seed, shift=shift)


def test_synthetic_goldens(gpu_ctx, golden):
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    config.set_precision(track="strict")
    imgs = _synth(0)
    tc = make_tc(max_residue=10.0, nPyramidLevels=3, subsampling=2)
    f = sgf.KLTSelectGoodFeatures(tc, imgs[0], 300)
    assert_features_equal(fl_arrays(f), fl(golden, "S640_sel300"))
    tf.KLTTrackFeatures(tc, imgs[0], imgs[1], f)
    assert_features_equal(fl_arrays(f), fl(golden, "S640_trk300"))
    imgs = _synth(1)
    tc = make_tc(window_width=15, window_height=15, nPyramidLevels=2, subsampling=4, max_residue=8.0)
    f = sgf.KLTSelectGoodFeatures(tc, imgs[0], 200)
    assert_features_equal(fl_arrays(f), fl(golden, "S640w15_sel200"))
    tf.KLTTrackFeatures(tc, imgs[0], imgs[1], f)
    assert_features_equal(fl_arrays(f), fl(golden, "S640w15_trk200"))
    # every status code
    imgs = _synth(2, (240, 320), (6.2, -9.4))
    tc = make_tc(nPyramidLevels=2, subsampling=2, max_residue=5.0, max_iterations=4, min_determinant=2000.0)
    f = sgf.KLTSelectGoodFeatures(tc, imgs[0], 150)
    assert_features_equal(fl_arrays(f), fl(golden, "H320_sel150"))
    tf.KLTTrackFeatures(tc, imgs[0], imgs[1], f)
    assert_features_equal(fl_arrays(f), fl(golden, "H320_trk150"))
    imgs = _synth(3, (240, 320))
    tc = make_tc(nPyramidLevels=2, subsampling=2, min_determinant=3.0e7)
    f = sgf.KLTSelectGoodFeatures(tc, imgs[0], 120)
    tf.KLTTrackFeatures(tc, imgs[0], imgs[1], f)
    assert_features_equal(fl_arrays(f), fl(golden, "D320_trk120"))


def test_patch_and_assert(gpu_ctx, golden):
    from pyfeaturetrack_b200 import trackFeaturesUtils
    assert np.array_equal(trackFeaturesUtils.extractImagePatchSlow(golden["A_smooth"], 100.3, 57.8, 7, 7), golden["A_patch"])
    with pytest.raises(AssertionError):
        trackFeaturesUtils.extractImagePatchSlow(golden["A_smooth"], 2.5, 57.8, 7, 7)


def test_feature_near_border_raises_like_reference(gpu_ctx, img01):
    from pyfeaturetrack_b200 import klt, trackFeatures as tf
    tc = make_tc()
    f = klt.KLT_Feature()
    f.x, f.y, f.val = 5.0, 100.0, 0       # window leaves the image at level 1: reference asserts (pyx:35)
    with pytest.raises(AssertionError):
        tf.KLTTrackFeatures(tc, img01[0], img01[1], [f])


# ---- full-size configs against the oracle -------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [dict(name="B", shape=(1080, 1920), n=1000, L=3, ss=2, w=7),
                                 dict(name="C", shape=(2160, 3840), n=10000, L=4, ss=2, w=7),
                                 dict(name="E-translational", shape=(1080, 1920), n=1000, L=3, ss=2, w=15)])
def test_full_size_configs(gpu_ctx, oracle, cfg):
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    H, W = cfg["shape"]
    imgs = _synth(0, (H, W))
    kw = dict(nPyramidLevels=cfg["L"], subsampling=cfg["ss"], window_width=cfg["w"], window_height=cfg["w"], max_residue=10.0)
    p = P(oracle, **kw)
    tc = make_tc(**kw)
    assert tc.borderx == p.borderx
    want_sel = oracle.select_good_features(p, imgs[0], cfg["n"])
    f = sgf.KLTSelectGoodFeatures(tc, imgs[0], cfg["n"])
    assert_features_equal(fl_arrays(f), want_sel)
    want_trk = oracle.track_features(p, imgs[0], imgs[1], *want_sel)[:3]
    config.set_precision(track="strict")
    tf.KLTTrackFeatures(tc, imgs[0], imgs[1], f)
    assert_features_equal(fl_arrays(f), want_trk)
    assert (want_trk[2] == 0).mean() > 0.95
    for mode in ("fast", "windowed"):
        config.set_precision(track=mode)
        f = sgf.KLTSelectGoodFeatures(tc, imgs[0], cfg["n"])
        tf.KLTTrackFeatures(tc, imgs[0], imgs[1], f)
        assert_features_close(fl_arrays(f), want_trk)


def test_batched_pairs_match_single(gpu_ctx, oracle):
    """klt_track_pairs_u8 over a batch of independent pairs == the same pairs one by one (the multi-GPU shard unit)."""
    from pyfeaturetrack_b200 import _capi, trackFeatures, selectGoodFeatures as sgf
    H, W, B, n = 240, 320, 4, 64
    tc = make_tc(nPyramidLevels=2, subsampling=2, max_residue=10.0)
    p = P(oracle, nPyramidLevels=2, subsampling=2, max_residue=10.0)
    f1 = np.empty((B, H, W), np.uint8)
    f2 = np.empty((B, H, W), np.uint8)
    xs = np.empty((B, n)); ys = np.empty((B, n)); vs = np.empty((B, n), np.int32)
    want = []
    for b in range(B):
        a, c = _synth(20 + b, (H, W))
        f1[b], f2[b] = a, c
        sel = oracle.select_good_features(p, a, n)
        xs[b], ys[b], vs[b] = sel
        want.append(oracle.track_features(p, a, c, *sel)[:3])
    taps = trackFeatures._taps_for_one_image(tc)
    params = sgf.make_params(tc)
    p1 = _capi.Pyramid(gpu_ctx, W, H, 2, 2, B)
    p2 = _capi.Pyramid(gpu_ctx, W, H, 2, 2, B)
    gpu_ctx.check(_capi.lib().klt_track_pairs_u8(gpu_ctx.handle, C.byref(params), C.byref(taps), _capi.PRECISION_STRICT,
                                                 p1.handle, p2.handle, f1.ctypes.data, f2.ctypes.data, W, W * H, n,
                                                 xs.ctypes.data, ys.ctypes.data, vs.ctypes.data))
    for b in range(B):
        assert_features_equal((xs[b], ys[b], vs[b]), want[b])
    p1.close(); p2.close()


def test_properties_full_size(gpu_ctx):
    """Size-independent properties at 1080p: identity tracking, idempotent selection, linearity of the convolution."""
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, convolve, config
    imgs = _synth(4, (1080, 1920))
    tc = make_tc(nPyramidLevels=3, subsampling=2, max_residue=10.0)
    f = sgf.KLTSelectGoodFeatures(tc, imgs[0], 1000)
    x0, y0, v0 = fl_arrays(f)
    assert (v0 > 0).all()
    d = np.maximum(np.abs(x0[:, None] - x0[None, :]), np.abs(y0[:, None] - y0[None, :]))
    np.fill_diagonal(d, 1e9)
    assert d.min() >= tc.mindist                      # Chebyshev min distance holds
    assert (np.diff(v0) <= 0).all()                   # best first
    g = sgf.KLTSelectGoodFeatures(tc, imgs[0], 1000)
    assert_features_equal(fl_arrays(g), (x0, y0, v0))   # deterministic
    tf.KLTTrackFeatures(tc, imgs[0], imgs[0], f)      # an image against itself: nothing moves, nothing is lost
    x1, y1, v1 = fl_arrays(f)
    assert (v1 == 0).all() and np.array_equal(x1, x0) and np.array_equal(y1, y0)
    config.set_precision(operator="fast")
    a = imgs[0].astype(np.float32)
    b = imgs[1].astype(np.float32)
    convolve._computeKernels(1.0)
    sa, sb, sab = (convolve.KLTComputeSmoothedImage(z, 1.0) for z in (a, b, a + b))
    assert np.abs(sab - (sa + sb)).max() <= 1e-4 * 510


# ---- affine consistency check (config E): parity against the in-repo C-KLT restatement, unpinned by the reference ----
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_affine_consistency_vs_restatement(gpu_ctx, oracle, mode):
    from test_oracle import _affine_sequence
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    config.set_precision(track="strict")          # identical translational results, so both affine trackers start equal
    frames = _affine_sequence()
    kw = dict(nPyramidLevels=2, subsampling=2, max_residue=10.0, affineConsistencyCheck=mode)
    p = P(oracle, **kw)
    tc = make_tc(**kw)
    p.borderx = p.bordery = tc.borderx = tc.bordery = max(p.borderx, 12.0)
    n = 150
    x, y, v = oracle.select_good_features(p, frames[0], n)
    aff = oracle.AffineState(n)
    f = sgf.KLTSelectGoodFeatures(tc, frames[0], n)
    assert_features_equal(fl_arrays(f), (x, y, v))
    for k in range(1, len(frames)):
        x, y, v, _ = oracle.track_features_affine(p, frames[k - 1], frames[k], x, y, v, aff)
        tf.KLTTrackFeatures(tc, frames[k - 1], frames[k], f)
        gx, gy, gv = fl_arrays(f)
        assert np.mean(gv == v) >= 0.99, (k, np.mean(gv == v))
        both = (gv == 0) & (v == 0)
        assert np.abs(gx[both] - x[both]).max() <= POS_TOL and np.abs(gy[both] - y[both]).max() <= POS_TOL
        gA = np.array([[ft.aff_Axx, ft.aff_Ayx, ft.aff_Axy, ft.aff_Ayy] for ft in f], np.float32)
        assert np.abs(gA[both] - aff.A[both]).max() <= 2e-3, (k, np.abs(gA[both] - aff.A[both]).max())
        gax = np.array([ft.aff_x for ft in f], np.float32)
        assert np.abs(gax[both] - aff.aff_x[both]).max() <= 1e-4
        has = np.array([ft.aff_img is not None for ft in f])
        assert np.array_equal(has[both], aff.has[both].astype(bool))
        # the oracle continues from ITS state; keep both sides on the oracle's features so that one flipped status
        # does not cascade (positions of commonly tracked features are identical in strict mode)
    t = np.asarray(f[int(np.flatnonzero(both)[0])].aff_img)
    assert t.shape == (17, 17)
    i = int(np.flatnonzero(both)[0])
    assert np.array_equal(t, aff.tmpl[i, 0])
    import pickle
    g = pickle.loads(pickle.dumps(f[i]))
    assert np.array_equal(np.asarray(g.aff_img), t)


def test_affine_large_config_E(gpu_ctx, oracle):
    """Config E shape: 1080p, 15x15 tracking windows, 15x15 affine windows, affineConsistencyCheck = 2."""
    from pyfeaturetrack_b200 import synth, selectGoodFeatures as sgf, trackFeatures as tf, config
    config.set_precision(track="strict")
    frames = synth.frames(1080, 1920, synth.sequence_shifts(3), seed=100)
    kw = dict(nPyramidLevels=3, subsampling=2, window_width=15, window_height=15, max_residue=10.0, affineConsistencyCheck=2,
              sequentialMode=True)
    p = P(oracle, **kw)
    tc = make_tc(**kw)
    n = 1000
    x, y, v = oracle.select_good_features(p, frames[0], n)
    aff = oracle.AffineState(n)
    f = sgf.KLTSelectGoodFeatures(tc, frames[0], n)
    state = {}
    for k in (1, 2):
        x, y, v, _ = oracle.track_features_affine(p, frames[k - 1], frames[k], x, y, v, aff, state)
        tf.KLTTrackFeatures(tc, frames[k - 1], frames[k], f)
        gx, gy, gv = fl_arrays(f)
        assert np.mean(gv == v) >= 0.995
        both = (gv == 0) & (v == 0)
        assert both.mean() > 0.9
        assert np.array_equal(gx[both], x[both]) and np.array_equal(gy[both], y[both])


# ---- operator-level shims of the reference's Cython modules ---------------------------------------------------------
def test_operator_level_iterate_and_patch_ops(gpu_ctx, oracle, golden, img01):
    import ctypes as C
    from pyfeaturetrack_b200 import trackFeaturesUtils as tfu, klt
    p = P(oracle, max_residue=10.0)
    pyr1, pyr2 = oracle.image_pyramids(p, img01[0]), oracle.image_pyramids(p, img01[1])
    tc = make_tc(max_residue=10.0)
    x, y, v = oracle.select_good_features(p, img01[0], 30)
    tp = oracle._track_params(p)
    for f in range(30):
        x1, y1 = float(x[f]), float(y[f])
        T = tfu.extractImagePatchSlow(pyr1[0][0], x1, y1, 7, 7)
        Tx = tfu.extractImagePatchSlow(pyr1[1][0], x1, y1, 7, 7)
        Ty = tfu.extractImagePatchSlow(pyr1[2][0], x1, y1, 7, 7)
        assert np.array_equal(T, oracle.extract_patch(pyr1[0][0], x1, y1, 7, 7))
        got = tfu.trackFeatureIterateCKLT(x1, y1, Tx, Ty, T, pyr2[0][0], pyr2[1][0], pyr2[2][0], tc)
        # oracle: one level, same start
        x2, y2, it = C.c_double(x1), C.c_double(y1), C.c_int()
        st = oracle.lib().orc_track_feature_level(x1, y1, C.byref(x2), C.byref(y2), oracle._f(pyr1[0][0]), oracle._f(pyr1[1][0]),
                                                  oracle._f(pyr1[2][0]), oracle._f(pyr2[0][0]), oracle._f(pyr2[1][0]),
                                                  oracle._f(pyr2[2][0]), 320, 240, C.byref(tp), C.byref(it))
        assert got[3] == it.value
        if got[2] == 0 and st in (0, -3, -5):      # the level wrapper adds the residue / max-iteration mapping on top
            assert (got[0], got[1]) == (x2.value, y2.value)
    # computeIntensityDifference / computeGradientSum
    work = np.empty((7, 7), np.float32)
    out = np.empty(49, np.float32)
    tfu.computeIntensityDifference(T, pyr2[0][0], 100.25, 80.5, work, out)
    want = (T - oracle.extract_patch(pyr2[0][0], 100.25, 80.5, 7, 7)).ravel()
    assert np.array_equal(out, want)
    jac = np.empty((49, 2), np.float32)
    tfu.computeGradientSum(Tx, pyr2[1][0], 100.25, 80.5, work, jac, 0)
    assert np.array_equal(jac[:, 0], (-Tx - oracle.extract_patch(pyr2[1][0], 100.25, 80.5, 7, 7)).ravel())


def test_enforce_minimum_distance_shim(gpu_ctx, oracle, golden, reference):
    """_enforceMinimumDistance on an explicit point list: the GPU shim against the reference's own Python function."""
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, klt
    rsgf, rklt = reference["selectGoodFeatures"], reference["klt"]
    val = golden["A_scan_val"]
    ys, xs = np.mgrid[30:210, 30:290]
    pts = sorted(zip(val.ravel().tolist(), xs.ravel().astype(np.int32), ys.ravel().astype(np.int32)))
    pts.reverse()
    pts = pts[:20000]
    for overwrite in (True, False):
        a = [klt.KLT_Feature() for _ in range(60)]
        b = [rklt.KLT_Feature() for _ in range(60)]
        if not overwrite:
            rng = np.random.default_rng(0)
            for fa, fb in zip(a, b):
                if rng.random() < 0.5:
                    fa.x = fb.x = float(rng.uniform(40, 280)); fa.y = fb.y = float(rng.uniform(40, 200)); fa.val = fb.val = 0
                else:
                    fa.x = fb.x = -1.0; fa.y = fb.y = -1.0; fa.val = fb.val = -4
        sgf._enforceMinimumDistance(pts, a, 320, 240, 10, 1, overwrite)
        rsgf._enforceMinimumDistance(pts, b, 320, 240, 10, 1, overwrite)
        assert [(float(f.x), float(f.y), int(f.val)) for f in a] == [(float(f.x), float(f.y), int(f.val)) for f in b]


def test_config_D_sequence_with_replacement(gpu_ctx, oracle):
    """Config D shape (shortened): one 1080p sequence in sequentialMode, per frame KLTTrackFeatures(prev, cur) then
    KLTReplaceLostFeatures; STRICT pyramids => bit-identical to the oracle frame after frame."""
    from pyfeaturetrack_b200 import synth, selectGoodFeatures as sgf, trackFeatures as tf, config
    config.set_precision(track="strict")
    nfr = 5
    shifts = [(s[0] * 6, s[1] * 6) for s in synth.sequence_shifts(nfr)]      # ~7 px/frame so that features get lost
    frames = synth.frames(1080, 1920, shifts, seed=101)
    kw = dict(nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    p = P(oracle, **kw)
    tc = make_tc(**kw)
    n = 1000
    x, y, v = oracle.select_good_features(p, frames[0], n)
    f = sgf.KLTSelectGoodFeatures(tc, frames[0], n)
    assert_features_equal(fl_arrays(f), (x, y, v))
    state = {}
    lost_total = 0
    for k in range(1, nfr):
        x, y, v, _ = oracle.track_features(p, frames[k - 1], frames[k], x, y, v, state)
        tf.KLTTrackFeatures(tc, frames[k - 1], frames[k], f)
        assert_features_equal(fl_arrays(f), (x, y, v))
        lost_total += int((v < 0).sum())
        _, gxs, gys = state["pyramid_last"]
        x, y, v, _ = oracle.select_from_gradients(p, gxs[0], gys[0], n, existing=(x, y, v))
        sgf.KLTReplaceLostFeatures(tc, frames[k], f)
        assert_features_equal(fl_arrays(f), (x, y, v))
        assert (v >= 0).all()
    assert lost_total > 0


# ---- more shapes: every window size the FAST kernel is instantiated for, several pyramid geometries, odd image sizes ----
@pytest.mark.parametrize("win,L,ss,shape", [(3, 2, 2, (200, 264)), (5, 3, 2, (240, 320)), (9, 2, 4, (241, 323)), (11, 1, 2, (180, 256)),
                                            (13, 2, 2, (256, 384)), (7, 2, 8, (360, 488)), (17, 2, 2, (300, 400)), (7, 4, 2, (480, 640))])
def test_tracking_window_and_pyramid_variants(gpu_ctx, oracle, win, L, ss, shape):
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    imgs = _synth(30 + win + L, shape, shift=(1.2, -1.9))
    kw = dict(window_width=win, window_height=win, nPyramidLevels=L, subsampling=ss, max_residue=12.0)
    p = P(oracle, **kw)
    tc = make_tc(**kw)
    assert p.borderx == tc.borderx
    n = 80
    want_sel = oracle.select_good_features(p, imgs[0], n)
    want_trk = oracle.track_features(p, imgs[0], imgs[1], *want_sel)[:3]
    for mode in ("strict", "fast", "windowed"):
        config.set_precision(track=mode)
        f = sgf.KLTSelectGoodFeatures(tc, imgs[0], n)
        assert_features_equal(fl_arrays(f), want_sel)
        tf.KLTTrackFeatures(tc, imgs[0], imgs[1], f)
        if mode == "strict":
            assert_features_equal(fl_arrays(f), want_trk)
        else:
            got = fl_arrays(f)
            assert np.mean(got[2] == want_trk[2]) >= 0.97          # 80 features: allow two threshold flips
            both = (got[2] == 0) & (want_trk[2] == 0)
            assert np.abs(got[0][both] - want_trk[0][both]).max() <= POS_TOL
            assert np.abs(got[1][both] - want_trk[1][both]).max() <= POS_TOL


@pytest.mark.parametrize("win,L,ss", [(3, 3, 2), (5, 3, 2), (9, 2, 4), (11, 2, 2), (13, 3, 2), (15, 2, 2)])
def test_window_sizes_at_1000_features(gpu_ctx, oracle, win, L, ss):
    """north_star's 99.9 % / 1e-3 px bar for every window size the windowed tracker is instantiated for (7x7: the full-size
    configs), on enough features for the fraction to mean something: 1000 features on 600x800 frames."""
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    imgs = _synth(70 + win, (600, 800), shift=(1.4, -0.8))
    kw = dict(window_width=win, window_height=win, nPyramidLevels=L, subsampling=ss, max_residue=10.0, mindist=8)
    p = P(oracle, **kw)
    tc = make_tc(**kw)
    n = 1000
    want_sel = oracle.select_good_features(p, imgs[0], n)
    assert (want_sel[2] >= 0).sum() >= 990
    want_trk = oracle.track_features(p, imgs[0], imgs[1], *want_sel)[:3]
    assert (want_trk[2] == 0).mean() > 0.9
    for mode in ("fast", "windowed"):
        config.set_precision(track=mode)
        f = sgf.KLTSelectGoodFeatures(tc, imgs[0], n)
        assert_features_equal(fl_arrays(f), want_sel)
        tf.KLTTrackFeatures(tc, imgs[0], imgs[1], f)
        got = fl_arrays(f)
        assert np.mean(got[2] == want_trk[2]) >= 0.999, (mode, win, float(np.mean(got[2] == want_trk[2])))
        both = (got[2] == 0) & (want_trk[2] == 0)
        assert np.abs(got[0][both] - want_trk[0][both]).max() <= POS_TOL
        assert np.abs(got[1][both] - want_trk[1][both]).max() <= POS_TOL


def test_random_feature_positions_and_dead_features(gpu_ctx, oracle):
    """Features the caller made up (fractional positions, some dead, some near the border): statuses follow the oracle."""
    from pyfeaturetrack_b200 import klt, trackFeatures as tf, config
    imgs = _synth(41, (300, 400), shift=(2.5, 3.5))
    kw = dict(nPyramidLevels=2, subsampling=2, max_residue=8.0)
    p = P(oracle, **kw)
    tc = make_tc(**kw)
    rng = np.random.default_rng(9)
    n = 400
    x = rng.uniform(16, 400 - 17, n).astype(np.float32).astype(np.float64)
    y = rng.uniform(16, 300 - 17, n).astype(np.float32).astype(np.float64)
    v = np.where(rng.random(n) < 0.2, rng.integers(-5, 0, n), rng.integers(0, 500, n)).astype(np.int32)
    want = oracle.track_features(p, imgs[0], imgs[1], x, y, v)[:3]
    for mode in ("strict", "fast", "windowed"):
        config.set_precision(track=mode)
        fl_ = []
        for i in range(n):
            f = klt.KLT_Feature(); f.x, f.y, f.val = float(x[i]), float(y[i]), int(v[i])
            fl_.append(f)
        tf.KLTTrackFeatures(tc, imgs[0], imgs[1], fl_)
        got = fl_arrays(fl_)
        dead = v < 0
        assert np.array_equal(got[2][dead], v[dead]) and np.array_equal(got[0][dead], x[dead])     # untouched
        if mode == "strict":
            assert_features_equal(got, want)
        else:
            assert_features_close(got, want)
    assert len(set(want[2].tolist())) >= 3
    # empty list and an all-dead list are no-ops
    tf.KLTTrackFeatures(tc, imgs[0], imgs[1], [])
    f = klt.KLT_Feature(); f.x, f.y, f.val = -1.0, -1.0, -4
    tf.KLTTrackFeatures(tc, imgs[0], imgs[1], [f])
    assert (f.x, f.y, f.val) == (-1.0, -1.0, -4)


def test_selection_edge_cases(gpu_ctx, oracle):
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf
    imgs = _synth(42, (160, 200))
    # more features requested than can exist at this mindist: the rest is KLT_NOT_FOUND (-1)
    kw = dict(mindist=25)
    p = P(oracle, **kw)
    tc = make_tc(**kw)
    want = oracle.select_good_features(p, imgs[0], 200)
    f = sgf.KLTSelectGoodFeatures(tc, imgs[0], 200)
    assert_features_equal(fl_arrays(f), want)
    assert (want[2] == -1).any() and (want[2] > 0).any()
    # mindist 0 / 1: no suppression; min_eigenvalue high: few features
    for kw in (dict(mindist=0), dict(mindist=1), dict(min_eigenvalue=4000), dict(nSkippedPixels=3, mindist=4)):
        p = P(oracle, **kw)
        tc = make_tc(**kw)
        assert_features_equal(fl_arrays(sgf.KLTSelectGoodFeatures(tc, imgs[0], 60)), oracle.select_good_features(p, imgs[0], 60))
    assert sgf.KLTSelectGoodFeatures(make_tc(), imgs[0], 0) == []


def test_windowed_pyramids_build_gradients_on_demand(gpu_ctx, oracle):
    """KLT_PRECISION_FAST_WINDOWED: image-only pyramids; a gradient plane asked for later equals the FAST build's, the
    windowed tracker agrees with the plane-based FAST tracker, and the affine tracker still works on such pyramids."""
    from pyfeaturetrack_b200 import _capi, trackFeatures, selectGoodFeatures as sgf
    H, W, L, ss, n = 360, 488, 3, 2, 300
    a, c = _synth(77, (H, W), shift=(2.2, -1.4))
    kw = dict(nPyramidLevels=L, subsampling=ss, max_residue=10.0)
    tc = make_tc(**kw)
    p = P(oracle, **kw)
    taps = trackFeatures._taps_for_one_image(tc)
    params = sgf.make_params(tc)
    sel = oracle.select_good_features(p, a, n)
    res = {}
    for name, prec in (("fast", _capi.PRECISION_FAST), ("windowed", _capi.PRECISION_FAST_WINDOWED)):
        p1 = _capi.Pyramid(gpu_ctx, W, H, L, ss, 1)
        p2 = _capi.Pyramid(gpu_ctx, W, H, L, ss, 1)
        p1.build_u8(a, taps, prec)
        p2.build_u8(c, taps, prec)
        x, y, v = (np.array(z) for z in sel)
        gpu_ctx.check(_capi.lib().klt_track_features(gpu_ctx.handle, C.byref(params), p1.handle, p2.handle, n,
                                                     x.ctypes.data, y.ctypes.data, v.ctypes.data, None))
        res[name] = (x, y, v, [p2.download(0, l) for l in range(L)], [p2.download(1, l) for l in range(L)],
                     [p2.download(2, l) for l in range(L)])
        p1.close(); p2.close()
    f, w = res["fast"], res["windowed"]
    for l in range(L):
        assert np.array_equal(f[3][l], w[3][l]) or np.abs(f[3][l] - w[3][l]).max() <= 1e-4      # same smoothing arithmetic
        for k in (4, 5):                                                                        # planes built on demand
            assert np.abs(f[k][l] - w[k][l]).max() <= 1e-5 * np.abs(f[k][l]).max()
    assert np.mean(f[2] == w[2]) >= 0.995
    both = (f[2] == 0) & (w[2] == 0)
    assert both.sum() > 0.8 * n
    assert np.abs(f[0][both] - w[0][both]).max() <= 1e-3 and np.abs(f[1][both] - w[1][both]).max() <= 1e-3
    want = oracle.track_features(p, a, c, *sel)[:3]
    assert_features_close((w[0], w[1], w[2]), want)


def test_windowed_sequence_and_affine(gpu_ctx, oracle):
    """sequentialMode (pyramid reuse) and the affine consistency check on image-only pyramids follow the FAST path."""
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    frames = [synth_frame(k) for k in range(4)]
    out = {}
    for mode in ("fast", "windowed"):
        for affine in (-1, 2):
            config.set_precision(track=mode)
            tc = make_tc(nPyramidLevels=2, subsampling=2, max_residue=10.0)
            tc.sequentialMode = True
            tc.affineConsistencyCheck = affine
            f = sgf.KLTSelectGoodFeatures(tc, frames[0], 120)
            for k in range(1, 4):                 # no replacement: one status flip would reshuffle every later slot
                tf.KLTTrackFeatures(tc, frames[k - 1], frames[k], f)
            out[(mode, affine)] = fl_arrays(f)
    for affine in (-1, 2):
        a, b = out[("fast", affine)], out[("windowed", affine)]
        assert np.mean(a[2] == b[2]) >= 0.97
        same = (a[2] == b[2])
        assert np.abs(a[0][same] - b[0][same]).max() <= 2e-3 and np.abs(a[1][same] - b[1][same]).max() <= 2e-3


def synth_frame(k, shape=(300, 400)):
    from pyfeaturetrack_b200 import synth
    base = _synth(5, (shape[0] + 16, shape[1] + 16))[0]
    return np.ascontiguousarray(base[k:k + shape[0], 2 * k:2 * k + shape[1]])


def test_windowed_large_motion_restages_its_region(gpu_ctx, oracle):
    """One pyramid level and a 3-4 px shift: the window walks out of the 2-pixel margin of the staged region during the
    Newton iterations, so the windowed tracker has to re-stage (and re-evaluate the gradients) mid-loop."""
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    imgs = _synth(91, (300, 400), shift=(3.6, -2.7))
    kw = dict(nPyramidLevels=1, subsampling=2, max_residue=15.0, max_iterations=20)
    p = P(oracle, **kw)
    tc = make_tc(**kw)
    n = 150
    want_sel = oracle.select_good_features(p, imgs[0], n)
    want = oracle.track_features(p, imgs[0], imgs[1], *want_sel)[:3]
    assert (want[2] == 0).mean() > 0.5                       # most features do converge across the 3-4 px
    moved = np.hypot(want[0] - want_sel[0], want[1] - want_sel[1])[want[2] == 0]
    assert np.median(moved) > 3.0
    out = {}
    for mode in ("fast", "windowed"):
        config.set_precision(track=mode)
        f = sgf.KLTSelectGoodFeatures(tc, imgs[0], n)
        tf.KLTTrackFeatures(tc, imgs[0], imgs[1], f)
        out[mode] = fl_arrays(f)
        got = out[mode]
        assert np.mean(got[2] == want[2]) >= 0.97
        both = (got[2] == 0) & (want[2] == 0)
        assert np.abs(got[0][both] - want[0][both]).max() <= POS_TOL and np.abs(got[1][both] - want[1][both]).max() <= POS_TOL
    assert np.mean(out["fast"][2] == out["windowed"][2]) >= 0.99


def test_windowed_sequence_replacement_reads_real_gradients(gpu_ctx, oracle):
    """KLTReplaceLostFeatures in sequentialMode selects on the tracking pyramid's level-0 gradients; on an image-only
    pyramid those planes must be built first (they were once left unwritten: replacement then filled too few slots)."""
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    frames = [synth_frame(k, (360, 480)) for k in range(3)]
    res = {}
    for mode in ("fast", "windowed"):
        config.set_precision(track=mode)
        tc = make_tc(nPyramidLevels=2, subsampling=2, max_residue=10.0)
        tc.sequentialMode = True
        f = sgf.KLTSelectGoodFeatures(tc, frames[0], 200)
        tf.KLTTrackFeatures(tc, frames[0], frames[1], f)
        for feat in f[::4]:                       # lose a quarter of the features on purpose
            feat.x, feat.y, feat.val = -1.0, -1.0, -3
        sgf.KLTReplaceLostFeatures(tc, frames[1], f)
        res[mode] = fl_arrays(f)
        if mode == "windowed":                    # the reference's tc.pyramid_last_gradx / _grady views keep working
            p = P(oracle, nPyramidLevels=2, subsampling=2)
            simg = oracle.smooth(frames[1].astype(np.float32), p.smooth_sigma(), p.cache)
            want_gx, want_gy = oracle.gradients(simg, p.grad_sigma, p.cache)
            got_gx, got_gy = tc.pyramid_last_gradx.img[0], tc.pyramid_last_grady.img[0]
            assert np.abs(got_gx - want_gx).max() <= 1e-5 * np.abs(want_gx).max()
            assert np.abs(got_gy - want_gy).max() <= 1e-5 * np.abs(want_gy).max()
            assert tc.pyramid_last_gradx.img[1].shape == (180, 240)      # coarser planes are built on demand as well
    for mode in res:
        assert (res[mode][2] >= 0).all()          # every lost slot was refilled
    a, b = res["fast"], res["windowed"]
    new_a = {(int(x), int(y)) for x, y, v in zip(*a) if v > 0}
    new_b = {(int(x), int(y)) for x, y, v in zip(*b) if v > 0}
    assert len(new_a) == len(new_b) >= 50         # the 50 slots lost on purpose + whatever tracking lost
    assert len(new_a & new_b) >= 0.9 * len(new_a)  # same gradients up to ~1e-6: the same corners win
    d = np.maximum(np.abs(b[0][:, None] - b[0][None, :]), np.abs(b[1][:, None] - b[1][None, :]))
    np.fill_diagonal(d, 1e9)
    assert d.min() >= tc.mindist - 1              # tracked positions are fractional: the integer grid test allows -1


def test_lighting_insensitive_vs_restatement(gpu_ctx, oracle):
    """tc.lighting_insensitive (the reference raises; restated from its commented C, parity UNPINNED): the exact-order
    kernel equals the oracle's restatement bit for bit on STRICT pyramids and within tolerance on FAST / image-only ones,
    and the mode does what it is for."""
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    a, b = _synth(5, (240, 320), shift=(1.6, -2.2))
    dim = np.clip(0.6 * b.astype(np.float32) + 40, 0, 255).astype(np.uint8)
    kw = dict(nPyramidLevels=2, subsampling=2, max_residue=10.0)
    p = P(oracle, lighting_insensitive=True, **kw)
    tc = make_tc(**kw)
    tc.lighting_insensitive = True
    n = 100
    sel = oracle.select_good_features(p, a, n)
    for img2 in (b, dim):
        want = oracle.track_features(p, a, img2, *sel)[:3]
        assert (want[2] == 0).sum() >= 80
        for mode in ("strict", "fast", "windowed"):
            config.set_precision(track=mode)
            f = sgf.KLTSelectGoodFeatures(tc, a, n)
            tf.KLTTrackFeatures(tc, a, img2, f)
            got = fl_arrays(f)
            if mode == "strict":
                assert_features_equal(got, want)
            else:
                assert np.mean(got[2] == want[2]) >= 0.98
                both = (got[2] == 0) & (want[2] == 0)
                assert np.abs(got[0][both] - want[0][both]).max() <= POS_TOL and np.abs(got[1][both] - want[1][both]).max() <= POS_TOL
    # without the normalisation the dimmed frame loses most features to KLT_LARGE_RESIDUE
    tc.lighting_insensitive = False
    config.set_precision(track="strict")
    f = sgf.KLTSelectGoodFeatures(tc, a, n)
    tf.KLTTrackFeatures(tc, a, dim, f)
    assert (fl_arrays(f)[2] == -5).sum() > 50
    # refused together with the affine check
    tc.lighting_insensitive = True
    tc.affineConsistencyCheck = 2
    with pytest.raises(Exception, match="Not implemented"):
        tf.KLTTrackFeatures(tc, a, dim, f)


def test_windowed_corner_configurations(gpu_ctx, oracle):
    """Image-only pyramids off the beaten path: float32 input images, a small image whose staged regions hang over the
    border (reflect path), a gradient kernel the windowed tracker does not serve (planes built on demand), and a batch
    of pairs through klt_track_pairs_u8."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf, trackFeatures as tf, config
    config.set_precision(track="windowed")
    # (1) float32 images (values off the uint8 grid)
    a, b = _synth(61, (240, 320), shift=(1.3, -0.8))
    af, bf = a.astype(np.float32) * 0.5 + 3.25, b.astype(np.float32) * 0.5 + 3.25
    kw = dict(nPyramidLevels=2, subsampling=2, max_residue=10.0)
    p, tc = P(oracle, **kw), make_tc(**kw)
    sel = oracle.select_good_features(p, af, 80)
    want = oracle.track_features(p, af, bf, *sel)[:3]
    f = sgf.KLTSelectGoodFeatures(tc, af, 80)
    tf.KLTTrackFeatures(tc, af, bf, f)
    got = fl_arrays(f)
    assert np.mean(got[2] == want[2]) >= 0.97
    both = (got[2] == 0) & (want[2] == 0)
    assert both.sum() > 60 and np.abs(got[0][both] - want[0][both]).max() <= POS_TOL
    # (2) small image, 3 levels: at the coarsest level (30 x 40) the staged 16 x 16 regions of the outer features hang over
    # the image border (reflected staging path)
    a, b = _synth(62, (120, 160), shift=(0.6, -0.4))
    kw = dict(nPyramidLevels=3, subsampling=2, max_residue=12.0, window_width=5, window_height=5)
    p, tc = P(oracle, **kw), make_tc(**kw)
    sel = oracle.select_good_features(p, a, 50)
    want = oracle.track_features(p, a, b, *sel)[:3]
    f = sgf.KLTSelectGoodFeatures(tc, a, 50)
    tf.KLTTrackFeatures(tc, a, b, f)
    got = fl_arrays(f)
    assert np.mean(got[2] == want[2]) >= 0.95
    both = (got[2] == 0) & (want[2] == 0)
    assert both.sum() >= 30 and np.abs(got[0][both] - want[0][both]).max() <= POS_TOL and np.abs(got[1][both] - want[1][both]).max() <= POS_TOL
    # (3) grad_sigma 1.5: 9- or 11-tap gradient kernels -> the windowed tracker declines, the planes are built on demand
    a, b = _synth(63, (240, 320), shift=(1.1, 1.4))
    kw = dict(nPyramidLevels=2, subsampling=2, max_residue=10.0, grad_sigma=1.5)
    p, tc = P(oracle, **kw), make_tc(**kw)
    sel = oracle.select_good_features(p, a, 80)
    want = oracle.track_features(p, a, b, *sel)[:3]
    f = sgf.KLTSelectGoodFeatures(tc, a, 80)
    tf.KLTTrackFeatures(tc, a, b, f)
    got = fl_arrays(f)
    assert np.mean(got[2] == want[2]) >= 0.97
    both = (got[2] == 0) & (want[2] == 0)
    assert np.abs(got[0][both] - want[0][both]).max() <= POS_TOL
    # (4) a batch of pairs in one call == the same pairs one at a time (bit for bit: same kernels, same data)
    H, W, B, n = 240, 320, 3, 64
    kw = dict(nPyramidLevels=2, subsampling=2, max_residue=10.0)
    p, tc = P(oracle, **kw), make_tc(**kw)
    taps, params = tf._taps_for_one_image(tc), sgf.make_params(tc)
    f1 = np.empty((B, H, W), np.uint8); f2 = np.empty((B, H, W), np.uint8)
    xs = np.empty((B, n)); ys = np.empty((B, n)); vs = np.empty((B, n), np.int32)
    for k in range(B):
        f1[k], f2[k] = _synth(70 + k, (H, W))
        xs[k], ys[k], vs[k] = oracle.select_good_features(p, f1[k], n)
    single = []
    for k in range(B):
        q1, q2 = _capi.Pyramid(gpu_ctx, W, H, 2, 2, 1), _capi.Pyramid(gpu_ctx, W, H, 2, 2, 1)
        x, y, v = xs[k].copy(), ys[k].copy(), vs[k].copy()
        gpu_ctx.check(_capi.lib().klt_track_pairs_u8(gpu_ctx.handle, C.byref(params), C.byref(taps), _capi.PRECISION_FAST_WINDOWED,
                                                     q1.handle, q2.handle, f1[k].ctypes.data, f2[k].ctypes.data, W, W * H, n,
                                                     x.ctypes.data, y.ctypes.data, v.ctypes.data))
        single.append((x, y, v)); q1.close(); q2.close()
    q1, q2 = _capi.Pyramid(gpu_ctx, W, H, 2, 2, B), _capi.Pyramid(gpu_ctx, W, H, 2, 2, B)
    gpu_ctx.check(_capi.lib().klt_track_pairs_u8(gpu_ctx.handle, C.byref(params), C.byref(taps), _capi.PRECISION_FAST_WINDOWED,
                                                 q1.handle, q2.handle, f1.ctypes.data, f2.ctypes.data, W, W * H, n,
                                                 xs.ctypes.data, ys.ctypes.data, vs.ctypes.data))
    for k in range(B):
        assert_features_equal((xs[k], ys[k], vs[k]), single[k])
        assert_features_close((xs[k], ys[k], vs[k]), oracle.track_features(p, f1[k], f2[k], *oracle.select_good_features(p, f1[k], n))[:3])
    q1.close(); q2.close()


def test_async_pairs_pipeline_matches_sync(gpu_ctx, oracle):
    """klt_track_pairs_u8_async: three different batches issued back to back on one context without waiting (the staging
    halves alternate, uploads overlap the previous call's kernels) give exactly the synchronous call's results; the
    sticky status word reports the reference's AssertionError case."""
    from pyfeaturetrack_b200 import _capi, trackFeatures as tf, selectGoodFeatures as sgf
    lib = _capi.lib()
    H, W, B, n, K = 240, 320, 2, 48, 3
    kw = dict(nPyramidLevels=2, subsampling=2, max_residue=10.0)
    p, tc = P(oracle, **kw), make_tc(**kw)
    taps, params = tf._taps_for_one_image(tc), sgf.make_params(tc)
    f1 = [gpu_ctx.pinned_array((B, H, W), np.uint8) for _ in range(K)]
    f2 = [gpu_ctx.pinned_array((B, H, W), np.uint8) for _ in range(K)]
    xs = [gpu_ctx.pinned_array((B, n), np.float64) for _ in range(K)]
    ys = [gpu_ctx.pinned_array((B, n), np.float64) for _ in range(K)]
    vs = [gpu_ctx.pinned_array((B, n), np.int32) for _ in range(K)]
    start = []
    for k in range(K):
        for b in range(B):
            f1[k][b], f2[k][b] = _synth(200 + 10 * k + b, (H, W), shift=(0.7 * (k + 1), -0.9 * (b + 1)))
            xs[k][b], ys[k][b], vs[k][b] = oracle.select_good_features(p, f1[k][b], n)
        start.append((xs[k].copy(), ys[k].copy(), vs[k].copy()))
    p1, p2 = _capi.Pyramid(gpu_ctx, W, H, 2, 2, B), _capi.Pyramid(gpu_ctx, W, H, 2, 2, B)
    for prec in (_capi.PRECISION_FAST_WINDOWED, _capi.PRECISION_STRICT):
        want = []
        for k in range(K):
            x, y, v = (a.copy() for a in start[k])
            gpu_ctx.check(lib.klt_track_pairs_u8(gpu_ctx.handle, C.byref(params), C.byref(taps), prec, p1.handle, p2.handle,
                                                 f1[k].ctypes.data, f2[k].ctypes.data, W, W * H, n, x.ctypes.data, y.ctypes.data, v.ctypes.data))
            want.append((x, y, v))
        for k in range(K):
            xs[k][:], ys[k][:], vs[k][:] = start[k]
        for k in range(K):
            gpu_ctx.check(lib.klt_track_pairs_u8_async(gpu_ctx.handle, C.byref(params), C.byref(taps), prec, p1.handle, p2.handle,
                                                       f1[k].ctypes.data, f2[k].ctypes.data, W, W * H, n, xs[k].ctypes.data,
                                                       ys[k].ctypes.data, vs[k].ctypes.data))
            gpu_ctx.check(lib.klt_async_mark(gpu_ctx.handle, k))
        gpu_ctx.check(lib.klt_async_wait(gpu_ctx.handle, 0))
        assert_features_equal((xs[0], ys[0], vs[0]), want[0])          # the first call is complete once its mark is reached
        gpu_ctx.check(lib.klt_async_result(gpu_ctx.handle))
        for k in range(K):
            assert_features_equal((xs[k], ys[k], vs[k]), want[k])
    # a feature whose window leaves a pyramid level: the synchronous call fails, the asynchronous one reports it later
    xs[0][:], ys[0][:], vs[0][:] = start[0]
    xs[0][0, 0], ys[0][0, 0], vs[0][0, 0] = 1.0, 1.0, 0
    assert lib.klt_track_pairs_u8_async(gpu_ctx.handle, C.byref(params), C.byref(taps), _capi.PRECISION_FAST_WINDOWED, p1.handle,
                                        p2.handle, f1[0].ctypes.data, f2[0].ctypes.data, W, W * H, n, xs[0].ctypes.data,
                                        ys[0].ctypes.data, vs[0].ctypes.data) == 0
    assert lib.klt_async_result(gpu_ctx.handle) == _capi.KLT_ERR_ASSERT
    assert lib.klt_async_result(gpu_ctx.handle) == 0                   # the status word is cleared by reading it
    p1.close(); p2.close()


def test_plain_c_demo_tracks_the_known_shift(gpu_ctx, tmp_path):
    """The C program of examples/ (select + klt_track_pairs_u8 through the bare ABI) recovers the (3, 2) pixel shift."""
    import re, subprocess, sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from test_capi_symbols import _build_c_demo
    r = subprocess.run([_build_c_demo(tmp_path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    m = re.match(r"tracked (\d+) of (\d+) features, median shift \(([-\d.]+), ([-\d.]+)\)", r.stdout)
    assert m, r.stdout
    assert int(m.group(1)) >= 0.8 * int(m.group(2))
    assert abs(float(m.group(3)) - 3.0) < 0.1 and abs(float(m.group(4)) - 2.0) < 0.1


@pytest.mark.gpu
def test_write_internal_images_dumps(gpu_ctx, oracle, img01, tmp_path, monkeypatch):
    """tc.writeInternalImages (selectGoodFeatures.py:201-204, trackFeatures.py:186-196): the dumps the reference names exist and
    hold the min/max-normalised planes (klt_util.py:6-34) of the images the oracle computes."""
    from PIL import Image
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf, trackFeatures as tf, config
    monkeypatch.chdir(tmp_path)
    config.set_precision(track="strict", select="strict")
    tc = make_tc(max_residue=10.0)
    tc.writeInternalImages = True
    fl = sgf.KLTSelectGoodFeatures(tc, img01[0], 50)
    tf.KLTTrackFeatures(tc, img01[0], img01[1], fl)
    tc.writeInternalImages = False
    names = ["kltimg_sgfrlf.pgm", "kltimg_sgfrlf_gx.pgm", "kltimg_sgfrlf_gy.pgm"]
    for i in range(int(tc.nPyramidLevels)):
        for tag in "ij":
            names += ["kltimg_tf_%s%d.pgm" % (tag, i), "kltimg_tf_%s%d_gx.pgm" % (tag, i), "kltimg_tf_%s%d_gy.pgm" % (tag, i)]
    for nme in names:
        assert (tmp_path / nme).exists(), nme
    p = P(oracle, max_residue=10.0)
    a0 = np.asarray(img01[0])
    smooth = oracle.smooth_image(p, a0) if hasattr(oracle, "smooth_image") else None
    got = np.array(Image.open(str(tmp_path / "kltimg_sgfrlf.pgm")))
    assert got.shape == a0.shape and got.min() == 0 and got.max() >= 254
    if smooth is not None:
        want = ((smooth - smooth.min()) * (255.0 / (smooth.max() - smooth.min()))).astype(np.uint8)
        assert np.abs(got.astype(int) - want.astype(int)).max() <= 1
