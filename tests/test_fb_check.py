"""Forward-backward consistency check (Kalal, Mikolajczyk, Matas, ICPR 2010; beyond the reference and C-KLT):
klt_track_features_fb, the check inside klt_sequence, and KLTTrackFeatures with tc.max_fb_error.

The reference is composed here from the oracle: the forward pass is oracle.track_on_pyramids from pyramid 1 to pyramid 2, the
backward pass the same call with the pyramids swapped on the forward result, and the decision is NumPy's
e = sqrt(dx*dx + dy*dy) in float64 against the threshold.  STRICT pyramids must reproduce it bit for bit (==)."""
import ctypes as C
import os

import numpy as np
import pytest

KLT_FB_ERROR = -6
BLOCK = (150, 278, 250, 378)          # rows [150, 278), columns [250, 378) of frame 2 come from another texture


# ---- reference composition -------------------------------------------------------------------------------------------------
def occluded_pair(seed, H=480, W=640):
    """Frame 2 = frame 1 shifted by (dy, dx) = (1.7, -3.3), with a 128 x 128 block replaced by the same region of another
    seed's texture."""
    from pyfeaturetrack_b200 import synth
    f1, f2 = synth.frame_pair(H, W, seed=seed)
    other = synth.frame_pair(H, W, seed=seed + 1000)[1]
    f2 = f2.copy()
    r0, r1, c0, c1 = BLOCK
    f2[r0:r1, c0:c1] = other[r0:r1, c0:c1]
    return f1, np.ascontiguousarray(f2)


def fb_reference(oracle, p, pyr1, pyr2, x, y, v, max_fb_error):
    """-> x, y, val, fb_error (float32), Newton iterations of both passes (None where a backward template left the image:
    the oracle gives no count for a call that raises)."""
    x0, y0 = np.array(x, np.float64), np.array(y, np.float64)
    xf, yf, vf, it = oracle.track_on_pyramids(p, pyr1, pyr2, x0, y0, v)
    try:
        xb, yb, vb, itb = oracle.track_on_pyramids(p, pyr2, pyr1, xf, yf, vf)
        it += itb
    except AssertionError:
        # the oracle raises for the whole call; the check rejects only the features whose window left the image
        it = None
        xb, yb, vb = xf.copy(), yf.copy(), vf.copy()
        for f in np.flatnonzero(vf == 0):
            try:
                a, b, c, _ = oracle.track_on_pyramids(p, pyr2, pyr1, xf[f:f + 1], yf[f:f + 1], vf[f:f + 1])
                xb[f], yb[f], vb[f] = a[0], b[0], c[0]
            except AssertionError:
                xb[f], yb[f], vb[f] = -1.0, -1.0, -4
    fwd = vf == 0
    done = fwd & (vb == 0)
    dx, dy = xb - x0, yb - y0
    e = np.sqrt(dx * dx + dy * dy)
    fb = np.where(done, e, -1.0).astype(np.float32)
    reject = fwd & ~(done & (e <= np.float64(np.float32(max_fb_error))))
    x_out, y_out, v_out = xf.copy(), yf.copy(), vf.copy()
    x_out[reject] = -1.0; y_out[reject] = -1.0; v_out[reject] = KLT_FB_ERROR
    return x_out, y_out, v_out, fb, it


def block_distance(x, y):
    """Distance of (x, y) from BLOCK (0 inside)."""
    r0, r1, c0, c1 = BLOCK
    ddx = np.maximum(np.maximum(c0 - x, x - (c1 - 1)), 0.0)
    ddy = np.maximum(np.maximum(r0 - y, y - (r1 - 1)), 0.0)
    return np.hypot(ddx, ddy)


def window_inside_block(x, y, hw=3):
    r0, r1, c0, c1 = BLOCK
    return (x - hw >= c0) & (x + hw <= c1 - 1) & (y - hw >= r0) & (y + hw <= r1 - 1)


def assertion_scene(oracle):
    """retain_trackers, 3 levels of subsampling 2, border 4, 240 x 320: features start at x = 20 and frame 2 is frame 1
    shifted 15 px left, so the forward pass ends near x = 5 and the backward template leaves level 2."""
    from pyfeaturetrack_b200 import synth
    f1, f2 = synth.frames(240, 320, [(0.0, 0.0), (0.0, -15.0)], seed=0)
    kw = dict(nPyramidLevels=3, subsampling=2, retainTrackers=True)
    p = oracle.Params(**kw)
    p.borderx = p.bordery = 4
    rows = np.array([60.0, 100.0, 140.0, 180.0])
    return f1, f2, kw, p, np.full(4, 20.0), rows, np.ones(4, np.int32)


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def test_fb_state_code_and_defaults():
    from pyfeaturetrack_b200 import klt, _capi
    assert klt.kltState.KLT_FB_ERROR == KLT_FB_ERROR
    assert klt.KLT_TrackingContext().max_fb_error is None
    for name in ("klt_track_features_fb", "klt_sequence_set_fb_check", "klt_sequence_get_fb_error"):
        assert name in _capi.SIGNATURES


def test_fb_header_declares_the_code():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with open(os.path.join(root, "include", "klt_b200.h")) as fh:
        assert "#define KLT_FB_ERROR (-6)" in fh.read()


@pytest.mark.parametrize("levels", [2, 3])
def test_fb_reference_rejects_the_occluded_block(oracle, levels):
    """On the oracle: at 1 px, at least half of the forward-tracked features whose window lies inside the replaced block are
    rejected, at most 2 % of those at least 8 px away from it, and the median distance away from it is below 0.03 px."""
    f1, f2 = occluded_pair(0)
    p = oracle.Params(nPyramidLevels=levels, subsampling=2)
    x, y, v = oracle.select_good_features(p, f1, 1000)
    pyr1, pyr2 = oracle.image_pyramids(p, f1), oracle.image_pyramids(p, f2)
    xf, yf, vf, _ = oracle.track_on_pyramids(p, pyr1, pyr2, x, y, v)
    gx, gy, gv, fb, _ = fb_reference(oracle, p, pyr1, pyr2, x, y, v, 1.0)
    fwd = vf == 0
    assert np.array_equal(gv[~fwd], vf[~fwd])                 # the check touches forward-tracked features only
    assert np.array_equal(gx[gv == 0], xf[gv == 0])           # survivors keep the forward result
    inside = fwd & window_inside_block(x, y)
    away = fwd & (block_distance(x, y) >= 8.0)
    rej = gv == KLT_FB_ERROR
    assert inside.sum() >= 20 and away.sum() >= 800
    assert rej[inside].mean() >= 0.5, (int(rej[inside].sum()), int(inside.sum()))
    assert rej[away].mean() <= 0.02, (int(rej[away].sum()), int(away.sum()))
    e_away = fb[away & (fb >= 0)]
    assert np.median(e_away) < 0.03
    assert (fb[~fwd] == -1.0).all()


def test_fb_reference_assertion_scene(oracle):
    """The oracle facts the assertion test relies on: rows 60, 140, 180 end the forward pass near x = 5 and their backward
    template leaves the image at level 2; row 100 drifts and comes back about 15 px away."""
    f1, f2, _, p, x, y, v = assertion_scene(oracle)
    pyr1, pyr2 = oracle.image_pyramids(p, f1), oracle.image_pyramids(p, f2)
    xf, yf, vf, _ = oracle.track_on_pyramids(p, pyr1, pyr2, x, y, v)
    assert (vf == 0).all()
    for f in (0, 2, 3):
        assert abs(xf[f] - 5.0) < 0.5, xf[f]
        with pytest.raises(AssertionError):
            oracle.track_on_pyramids(p, pyr2, pyr1, xf[f:f + 1], yf[f:f + 1], vf[f:f + 1])
    xb, yb, vb, _ = oracle.track_on_pyramids(p, pyr2, pyr1, xf[1:2], yf[1:2], vf[1:2])
    assert vb[0] == 0 and np.hypot(xb[0] - 20.0, yb[0] - 100.0) > 10.0
    gx, gy, gv, fb, it = fb_reference(oracle, p, pyr1, pyr2, x, y, v, 1.0)
    assert (gv == KLT_FB_ERROR).all() and it is None
    assert fb[1] > 10.0 and (fb[[0, 2, 3]] == -1.0).all()


# ---- GPU -------------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture
def _quiet():
    from pyfeaturetrack_b200 import selectGoodFeatures, trackFeatures, config
    selectGoodFeatures.KLT_verbose = 0
    trackFeatures.KLT_verbose = 0
    yield
    config.set_precision(track="fast", select="strict", operator="strict")


def make_tc(**kw):
    from pyfeaturetrack_b200 import klt
    tc = klt.KLT_TrackingContext()
    for k, val in kw.items():
        setattr(tc, k, val)
    tc.KLTUpdateTCBorder()
    return tc


def build_batch(ctx, tc, frames, precision):
    from pyfeaturetrack_b200 import _capi, trackFeatures as tf
    H, W = frames[0].shape
    pyr = _capi.Pyramid(ctx, W, H, int(tc.nPyramidLevels), int(tc.subsampling), len(frames))
    pyr.build_u8(np.ascontiguousarray(np.stack(frames)), tf._taps_for_one_image(tc), precision)
    return pyr


def track_fb(ctx, tc, pyr1, pyr2, x, y, v, max_fb_error, device=False, plain=False):
    """klt_track_features_fb (plain: klt_track_features) on [batch][n] arrays -> x, y, val, fb_error, n_iterations"""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf
    lib = _capi.lib()
    params = sgf.make_params(tc)
    x, y, v = np.array(x, np.float64), np.array(y, np.float64), np.array(v, np.int32)
    fb = np.full(x.shape, 7.0, np.float32)
    n = x.shape[-1]
    it = C.c_int64()
    if device:
        d = [ctx.device_alloc(a.nbytes) for a in (x, y, v, fb)]
        for dst, a in zip(d, (x, y, v)):
            ctx.memcpy(dst, a, a.nbytes)
        args = d
    else:
        args = [a.ctypes.data for a in (x, y, v, fb)]
    if plain:
        ctx.check(lib.klt_track_features(ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, n, args[0], args[1], args[2],
                                         C.byref(it)))
    else:
        ctx.check(lib.klt_track_features_fb(ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, n, max_fb_error, args[0],
                                            args[1], args[2], args[3], C.byref(it)))
    if device:
        for src, a in zip(args, (x, y, v, fb)):
            ctx.memcpy(a, src, a.nbytes)
        ctx.sync()
        for p in args:
            ctx.device_free(p)
    return x, y, v, fb, it.value


def eq(got, want):
    for a, b in zip(got, want):
        assert np.array_equal(np.asarray(a), np.asarray(b))


@gpu
@pytest.mark.parametrize("levels", [2, 3])
def test_fb_strict_equals_the_oracle_composition(gpu_ctx, oracle, _quiet, levels):
    """STRICT pyramids, 3 occluded pairs in one batch, thresholds 0.1 and 1.0 px, host and device arrays: x, y, val and
    fb_error == the composed oracle; n_iterations counts both passes."""
    from pyfeaturetrack_b200 import _capi
    kw = dict(nPyramidLevels=levels, subsampling=2)
    tc, p = make_tc(**kw), oracle.Params(**kw)
    pairs = [occluded_pair(s) for s in range(3)]
    n = 1000
    sel = [oracle.select_good_features(p, f1, n) for f1, _ in pairs]
    x, y, v = (np.stack([s[i] for s in sel]) for i in range(3))
    pyr1 = build_batch(gpu_ctx, tc, [a for a, _ in pairs], _capi.PRECISION_STRICT)
    pyr2 = build_batch(gpu_ctx, tc, [b for _, b in pairs], _capi.PRECISION_STRICT)
    opyr = [(oracle.image_pyramids(p, a), oracle.image_pyramids(p, b)) for a, b in pairs]
    rejected = 0
    for thr in (0.1, 1.0):
        want = [fb_reference(oracle, p, o1, o2, x[b], y[b], v[b], thr) for b, (o1, o2) in enumerate(opyr)]
        for device in (False, True):
            gx, gy, gv, gfb, it = track_fb(gpu_ctx, tc, pyr1, pyr2, x, y, v, thr, device=device)
            for b in range(3):
                eq((gx[b], gy[b], gv[b], gfb[b]), want[b][:4])
            if all(w[4] is not None for w in want):
                assert it == sum(w[4] for w in want)
        rejected += int((gv == KLT_FB_ERROR).sum())
    assert rejected > 0
    pyr1.close(); pyr2.close()


@gpu
def test_fb_lighting_insensitive_strict(gpu_ctx, oracle, _quiet):
    """lighting_insensitive runs the exact-order kernel both ways: == the composed oracle in that mode."""
    from pyfeaturetrack_b200 import _capi
    kw = dict(nPyramidLevels=2, subsampling=2, lighting_insensitive=True)
    tc, p = make_tc(**kw), oracle.Params(**kw)
    f1, f2 = occluded_pair(4)
    x, y, v = oracle.select_good_features(p, f1, 500)
    pyr1, pyr2 = build_batch(gpu_ctx, tc, [f1], _capi.PRECISION_STRICT), build_batch(gpu_ctx, tc, [f2], _capi.PRECISION_STRICT)
    want = fb_reference(oracle, p, oracle.image_pyramids(p, f1), oracle.image_pyramids(p, f2), x, y, v, 1.0)
    for device in (False, True):
        got = track_fb(gpu_ctx, tc, pyr1, pyr2, x[None], y[None], v[None], 1.0, device=device)
        eq((got[0][0], got[1][0], got[2][0], got[3][0]), want[:4])
    assert (want[2] == KLT_FB_ERROR).any()
    pyr1.close(); pyr2.close()


@gpu
def test_fb_rejects_invalid_thresholds(gpu_ctx, _quiet):
    from pyfeaturetrack_b200 import _capi, synth, selectGoodFeatures as sgf, trackFeatures as tf
    tc = make_tc(nPyramidLevels=2, subsampling=2)
    f1 = synth.frames(240, 320, [(0.0, 0.0)], seed=3)[0]
    pyr = build_batch(gpu_ctx, tc, [f1], _capi.PRECISION_FAST)
    params = sgf.make_params(tc)
    x, y, v = np.array([160.0]), np.array([120.0]), np.zeros(1, np.int32)
    for bad in (0.0, -1.0, float("nan"), float("inf")):
        rc = _capi.lib().klt_track_features_fb(gpu_ctx.handle, C.byref(params), pyr.handle, pyr.handle, 1, bad, x.ctypes.data,
                                               y.ctypes.data, v.ctypes.data, None, None)
        assert rc == _capi.KLT_ERR_INVALID, bad
    q = _capi.Sequence(gpu_ctx, params, tf._taps_for_one_image(tc), 320, 240, 1, 10, _capi.PRECISION_FAST, _capi.SELECT_STRICT)
    for bad in (-1.0, float("nan"), float("inf")):
        assert _capi.lib().klt_sequence_set_fb_check(gpu_ctx.handle, q.handle, bad) == _capi.KLT_ERR_INVALID
    q.close()
    pyr.close()


@gpu
@pytest.mark.parametrize("precision,tracker", [("fast", "lk_track_rows"), ("windowed", "lk_windowed")])
def test_fb_fast_modes_track_the_strict_composition(gpu_ctx, oracle, _quiet, precision, tracker):
    """FAST pyramids (lk_track_rows) and image-only pyramids (lk_windowed): both passes run the same kernel, fb_prepare and
    fb_check once each; fb_error within 2e-3 px of the STRICT composition where both tracked, and the decisions agree except
    where the STRICT distance lies within 2e-3 px of the threshold or the forward statuses differ (under 1 % together)."""
    from pyfeaturetrack_b200 import _capi
    prec = dict(fast=_capi.PRECISION_FAST, windowed=_capi.PRECISION_FAST_WINDOWED)[precision]
    kw = dict(nPyramidLevels=3, subsampling=2)
    tc, p = make_tc(**kw), oracle.Params(**kw)
    pairs = [occluded_pair(s) for s in range(3)]
    n, thr = 1000, 1.0
    sel = [oracle.select_good_features(p, f1, n) for f1, _ in pairs]
    x, y, v = (np.stack([s[i] for s in sel]) for i in range(3))
    pyr1 = build_batch(gpu_ctx, tc, [a for a, _ in pairs], prec)
    pyr2 = build_batch(gpu_ctx, tc, [b for _, b in pairs], prec)
    gpu_ctx.profile(True)
    gpu_ctx.profile_reset()
    try:
        gx, gy, gv, gfb, _ = track_fb(gpu_ctx, tc, pyr1, pyr2, x, y, v, thr)
        kernels = gpu_ctx.profile_read()
    finally:
        gpu_ctx.profile(False)
    assert [k for k in ("lk_windowed", "lk_track_rows", "lk_track") if k in kernels] == [tracker], sorted(kernels)
    assert kernels[tracker]["launches"] == 2
    assert kernels["fb_prepare"]["launches"] == 1 and kernels["fb_check"]["launches"] == 1
    fwd_fast = track_fb(gpu_ctx, tc, pyr1, pyr2, x, y, v, thr, plain=True)[2]
    worst, excused, wrong, total = 0.0, 0, 0, 0
    for b, (f1, f2) in enumerate(pairs):
        o1, o2 = oracle.image_pyramids(p, f1), oracle.image_pyramids(p, f2)
        _, _, wv, wfb, _ = fb_reference(oracle, p, o1, o2, x[b], y[b], v[b], thr)
        wfwd = oracle.track_on_pyramids(p, o1, o2, x[b], y[b], v[b])[2]
        both = (wfb >= 0) & (gfb[b] >= 0)
        worst = max(worst, float(np.abs(gfb[b][both].astype(np.float64) - wfb[both]).max()))
        differ = (gv[b] == KLT_FB_ERROR) != (wv == KLT_FB_ERROR)
        near = (wfb >= 0) & (np.abs(wfb.astype(np.float64) - thr) <= 2e-3)
        ex = near | (fwd_fast[b] != wfwd)
        wrong += int((differ & ~ex).sum())
        excused += int(ex.sum())
        total += n
    assert worst <= 2e-3, worst
    assert wrong == 0
    assert excused < 0.01 * total, excused
    assert (gv == KLT_FB_ERROR).any()
    pyr1.close(); pyr2.close()


@gpu
@pytest.mark.parametrize("precision", ["strict", "fast", "windowed"])
def test_fb_backward_window_leaving_the_image_rejects_without_assert(gpu_ctx, oracle, _quiet, precision):
    """A backward template that leaves the image rejects the feature (KLT_FB_ERROR) and raises nothing, immediately or at
    klt_sync; the same features through klt_track_features come back tracked.  The drifting feature is rejected on e."""
    from pyfeaturetrack_b200 import _capi
    prec = dict(strict=_capi.PRECISION_STRICT, fast=_capi.PRECISION_FAST, windowed=_capi.PRECISION_FAST_WINDOWED)[precision]
    f1, f2, kw, p, x, y, v = assertion_scene(oracle)
    tc = make_tc(**kw)
    tc.borderx = tc.bordery = 4
    pyr1, pyr2 = build_batch(gpu_ctx, tc, [f1], prec), build_batch(gpu_ctx, tc, [f2], prec)
    for device in (False, True):
        gx, gy, gv, gfb, _ = track_fb(gpu_ctx, tc, pyr1, pyr2, x[None], y[None], v[None], 1.0, device=device)
        assert (gv == KLT_FB_ERROR).all() and (gx == -1.0).all() and (gy == -1.0).all()
        assert gfb[0][1] > 10.0 and (gfb[0][[0, 2, 3]] == -1.0).all()
    # deferred: device arrays without n_iterations only enqueue; the backward pass must not raise the sticky flag
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf
    params = sgf.make_params(tc)
    d = [gpu_ctx.device_alloc(32), gpu_ctx.device_alloc(32), gpu_ctx.device_alloc(16)]
    for dst, a in zip(d, (x, y, v)):
        gpu_ctx.memcpy(dst, a, a.nbytes)
    gpu_ctx.check(_capi.lib().klt_track_features_fb(gpu_ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, 4, 1.0, d[0], d[1],
                                                    d[2], None, None))
    assert _capi.lib().klt_sync(gpu_ctx.handle) == 0
    for a in d:
        gpu_ctx.device_free(a)
    px, py, pv, _, _ = track_fb(gpu_ctx, tc, pyr1, pyr2, x[None], y[None], v[None], 1.0, plain=True)
    assert (pv == 0).all()
    if precision == "strict":
        want = oracle.track_on_pyramids(p, oracle.image_pyramids(p, f1), oracle.image_pyramids(p, f2), x, y, v)
        eq((px[0], py[0], pv[0]), want[:3])
    pyr1.close(); pyr2.close()


@gpu
def test_fb_dropin_and_replacement(gpu_ctx, oracle, _quiet):
    """KLTTrackFeatures with tc.max_fb_error == the composed oracle (STRICT); in sequentialMode KLTReplaceLostFeatures refills
    the rejected slots; with the affine check it raises like lighting_insensitive does."""
    from pyfeaturetrack_b200 import config, selectGoodFeatures as sgf, trackFeatures as tf, klt
    config.set_precision(track="strict", select="strict")
    kw = dict(nPyramidLevels=3, subsampling=2)
    f1, f2 = occluded_pair(1)
    p = oracle.Params(**kw)
    for sequential in (False, True):
        tc = make_tc(sequentialMode=sequential, **kw)
        tc.max_fb_error = 1.0
        fl = sgf.KLTSelectGoodFeatures(tc, f1, 600)
        x = np.array([float(f.x) for f in fl]); y = np.array([float(f.y) for f in fl]); v = np.array([f.val for f in fl], np.int32)
        tf.KLTTrackFeatures(tc, f1, f2, fl)
        got = (np.array([float(f.x) for f in fl]), np.array([float(f.y) for f in fl]), np.array([f.val for f in fl], np.int32))
        want = fb_reference(oracle, p, oracle.image_pyramids(p, f1), oracle.image_pyramids(p, f2), x, y, v, 1.0)
        eq(got, want[:3])
        rej = got[2] == klt.kltState.KLT_FB_ERROR
        assert rej.any()
        if sequential:
            sgf.KLTReplaceLostFeatures(tc, f2, fl)
            after = np.array([f.val for f in fl])
            assert (after[rej] > 0).all()
    tc = make_tc(affineConsistencyCheck=0, **kw)
    tc.max_fb_error = 1.0
    fl = sgf.KLTSelectGoodFeatures(tc, f1, 50)
    with pytest.raises(Exception, match="Not implemented"):
        tf.KLTTrackFeatures(tc, f1, f2, fl)


# ---- sequences -------------------------------------------------------------------------------------------------------------
def occluded_sequence(H, W, nframes, seed):
    """A sequence of the shifted texture with a 96 x 96 block of another texture moving across it."""
    from pyfeaturetrack_b200 import synth
    shifts = [(s[0] * 5.0, s[1] * 5.0) for s in synth.sequence_shifts(nframes)]
    frames = synth.frames(H, W, shifts, seed=seed)
    other = synth.frames(H, W, [(0.0, 0.0)], seed=seed + 1000)[0]
    out = []
    for k, f in enumerate(frames):
        f = f.copy()
        r, c = 120 + 4 * k, 200 + 7 * k
        f[r:r + 96, c:c + 96] = other[r:r + 96, c:c + 96]
        out.append(np.ascontiguousarray(f))
    return out


def oracle_fb_sequence(oracle, p, frames, n, fb_on):
    """select, then per frame: track (sequentialMode), the FB step where fb_on(k), replacement on pyramid_last's gradients.
    -> per frame (x, y, val, val_tracked, fb_error)"""
    pyr = oracle.image_pyramids(p, frames[0])
    x, y, v, _ = oracle.select_from_gradients(p, pyr[1][0], pyr[2][0], n)
    out = [(x.copy(), y.copy(), v.copy(), None, None)]
    for k in range(1, len(frames)):
        cur = oracle.image_pyramids(p, frames[k])
        if fb_on(k):
            x, y, v, fb, _ = fb_reference(oracle, p, pyr, cur, x, y, v, 0.5)
        else:
            x, y, v, _ = oracle.track_on_pyramids(p, pyr, cur, x, y, v)
            fb = np.full(n, -1.0, np.float32)
        vt = v.copy()
        x, y, v, _ = oracle.select_from_gradients(p, cur[1][0], cur[2][0], n, existing=(x, y, v))
        out.append((x.copy(), y.copy(), v.copy(), vt, fb))
        pyr = cur
    return out


def run_fb_sequence(ctx, tc, seqs, n, off_at=None):
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf, trackFeatures as tf
    B, nfr = len(seqs), len(seqs[0])
    H, W = seqs[0][0].shape
    q = _capi.Sequence(ctx, sgf.make_params(tc), tf._taps_for_one_image(tc), W, H, B, n, _capi.PRECISION_STRICT,
                       _capi.SELECT_STRICT)
    q.start(np.ascontiguousarray(np.stack([s[0] for s in seqs])))
    q.set_fb_check(0.5)
    out = [q.features() + (None,)]
    for k in range(1, nfr):
        if k == off_at:
            q.set_fb_check(0)
        q.step(np.ascontiguousarray(np.stack([s[k] for s in seqs])))
        out.append(q.features() + (q.fb_error(),))
    iters = q.sync()
    graph = q.uses_graph()
    q.close()
    return out, graph, iters


@gpu
def test_fb_sequence_strict_equals_oracle(gpu_ctx, oracle, _quiet, monkeypatch):
    """STRICT + STRICT klt_sequence with set_fb_check(0.5), 4 sequences x 15 frames, replacement, CUDA graphs: after every step
    x, y, val, val_tracked and fb_error == the oracle sequence with the FB step before replacement; the plain-launch run is
    identical; set_fb_check(0) at step 8 gives, from then on, what the sequence without the check gives."""
    kw = dict(nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    tc, p = make_tc(**kw), oracle.Params(**kw)
    n, nfr, nseq = 300, 15, 4
    seqs = [occluded_sequence(480, 640, nfr, 200 + s) for s in range(nseq)]
    monkeypatch.delenv("KLT_B200_NO_GRAPH", raising=False)
    got, graph, _ = run_fb_sequence(gpu_ctx, tc, seqs, n)
    assert graph
    monkeypatch.setenv("KLT_B200_NO_GRAPH", "1")
    plain, graph2, _ = run_fb_sequence(gpu_ctx, tc, seqs, n)
    assert not graph2
    for k in range(nfr):
        for a, b in zip(got[k], plain[k]):
            assert (a is None and b is None) or np.array_equal(a, b), k
    monkeypatch.delenv("KLT_B200_NO_GRAPH", raising=False)
    off, _, _ = run_fb_sequence(gpu_ctx, tc, seqs, n, off_at=8)
    rejected = 0
    for s in range(nseq):
        for run, fb_on in ((got, lambda k: True), (off, lambda k: k < 8)):
            want = oracle_fb_sequence(oracle, p, seqs[s], n, fb_on)
            for k in range(nfr):
                gx, gy, gv, gvt, gfb = run[k]
                eq((gx[s], gy[s], gv[s]), want[k][:3])
                if k:
                    assert np.array_equal(gvt[s], want[k][3]), (s, k)
                    assert np.array_equal(gfb[s], want[k][4]), (s, k)
                    if run is got:
                        rejected += int((want[k][3] == KLT_FB_ERROR).sum())
    assert rejected > 0
