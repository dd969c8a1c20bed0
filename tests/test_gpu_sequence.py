"""GPU parity tests of the batched, synchronisation-free selection chain and of klt_sequence (BASELINE config D): the CUDA
path through the C ABI against the CPU oracle on the same seeded inputs.  STRICT = bit-exact (==); FAST = set overlap /
tolerances as north_star states them."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _quiet():
    from pyfeaturetrack_b200 import selectGoodFeatures, trackFeatures, config
    selectGoodFeatures.KLT_verbose = 0
    trackFeatures.KLT_verbose = 0
    config.set_precision(track="fast", select="strict", operator="strict")
    yield
    config.set_precision(track="fast", select="strict", operator="strict")


def make_tc(**kw):
    from pyfeaturetrack_b200 import klt
    tc = klt.KLT_TrackingContext()
    for k, v in kw.items():
        setattr(tc, k, v)
    tc.KLTUpdateTCBorder()
    return tc


def eq(got, want):
    assert np.array_equal(np.asarray(got[2], np.int64), np.asarray(want[2], np.int64))
    assert np.array_equal(np.asarray(got[0], np.float64), np.asarray(want[0], np.float64))
    assert np.array_equal(np.asarray(got[1], np.float64), np.asarray(want[1], np.float64))


def build_batch(ctx, tc, frames, precision):
    """frames: list of uint8 (H, W) -> a pyramid batch built like ComputeImagePyramids builds one image."""
    from pyfeaturetrack_b200 import _capi, trackFeatures as tf
    H, W = frames[0].shape
    pyr = _capi.Pyramid(ctx, W, H, int(tc.nPyramidLevels), int(tc.subsampling), len(frames))
    pyr.build_u8(np.ascontiguousarray(np.stack(frames)), tf._taps_for_one_image(tc), precision)
    return pyr


def batch_select(ctx, tc, pyr, n, replace, mode, x=None, y=None, v=None):
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf
    B = pyr.batch
    if x is None:
        x, y, v = np.full((B, n), -1.0), np.full((B, n), -1.0), np.full((B, n), -1, np.int32)
    else:
        x, y, v = np.array(x, np.float64), np.array(y, np.float64), np.array(v, np.int32)
    params = sgf.make_params(tc)
    ctx.check(_capi.lib().klt_select_good_features_batch(ctx.handle, C.byref(params), pyr.handle, n, 1 if replace else 0, mode,
                                                        x.ctypes.data, y.ctypes.data, v.ctypes.data))
    return x, y, v


def oracle_select_on_pyramid(oracle, p, frame, n, existing=None):
    _, gxs, gys = oracle.image_pyramids(p, frame)
    return oracle.select_from_gradients(p, gxs[0], gys[0], n, existing=existing)[:3]


# ---- batched selection ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,n,B,kw", [((240, 320), 100, 3, dict()),
                                          ((480, 640), 300, 4, dict(nPyramidLevels=3, subsampling=2)),
                                          ((243, 325), 80, 2, dict(nSkippedPixels=1, mindist=6)),
                                          ((300, 400), 120, 2, dict(window_width=15, window_height=15, nPyramidLevels=2, subsampling=2)),
                                          ((1080, 1920), 1000, 2, dict(nPyramidLevels=3, subsampling=2))])
def test_batch_select_strict_equals_oracle(gpu_ctx, oracle, shape, n, B, kw):
    """klt_select_good_features_batch (SELECTING_ALL, then REPLACING_SOME after knocking features out) == the oracle for
    every image of the batch, slots included."""
    from pyfeaturetrack_b200 import _capi, synth
    tc = make_tc(**kw)
    p = oracle.Params(**kw)
    frames = [synth.frames(shape[0], shape[1], [(0.0, 0.0)], seed=40 + s)[0] for s in range(B)]
    pyr = build_batch(gpu_ctx, tc, frames, _capi.PRECISION_STRICT)
    x, y, v = batch_select(gpu_ctx, tc, pyr, n, False, _capi.SELECT_STRICT)
    want = [oracle_select_on_pyramid(oracle, p, f, n) for f in frames]
    for b in range(B):
        eq((x[b], y[b], v[b]), want[b])
    # replacement: lose a different subset per image (also none / all), move the survivors a little (non-integer positions)
    rng = np.random.default_rng(5)
    x2, y2, v2 = x.copy(), y.copy(), v.copy()
    for b in range(B):
        frac = [0.05, 0.0, 1.0, 0.5][b % 4]
        lost = rng.random(n) < frac
        live = v2[b] >= 0
        x2[b][live] += rng.uniform(-0.9, 0.9, int(live.sum()))
        y2[b][live] += rng.uniform(-0.9, 0.9, int(live.sum()))
        x2[b][lost] = -1.0; y2[b][lost] = -1.0; v2[b][lost] = -4
        v2[b][~lost & live] = 0
    gx, gy, gv = batch_select(gpu_ctx, tc, pyr, n, True, _capi.SELECT_STRICT, x2, y2, v2)
    for b in range(B):
        eq((gx[b], gy[b], gv[b]), oracle_select_on_pyramid(oracle, p, frames[b], n, existing=(x2[b], y2[b], v2[b])))
    pyr.close()


def test_batch_select_device_arrays_no_sync(gpu_ctx, oracle):
    """Device-resident feature lists: the call only enqueues; results equal the host-array call."""
    from pyfeaturetrack_b200 import _capi, synth, selectGoodFeatures as sgf
    kw = dict(nPyramidLevels=2, subsampling=2)
    tc = make_tc(**kw)
    frames = [synth.frames(240, 320, [(0.0, 0.0)], seed=7 + s)[0] for s in range(3)]
    pyr = build_batch(gpu_ctx, tc, frames, _capi.PRECISION_STRICT)
    n, B = 90, 3
    hx, hy, hv = batch_select(gpu_ctx, tc, pyr, n, False, _capi.SELECT_STRICT)
    dx, dy, dv = gpu_ctx.device_alloc(B * n * 8), gpu_ctx.device_alloc(B * n * 8), gpu_ctx.device_alloc(B * n * 4)
    params = sgf.make_params(tc)
    gpu_ctx.check(_capi.lib().klt_select_good_features_batch(gpu_ctx.handle, C.byref(params), pyr.handle, n, 0, _capi.SELECT_STRICT, dx, dy, dv))
    x, y, v = np.empty((B, n)), np.empty((B, n)), np.empty((B, n), np.int32)
    gpu_ctx.memcpy(x, dx, B * n * 8); gpu_ctx.memcpy(y, dy, B * n * 8); gpu_ctx.memcpy(v, dv, B * n * 4)
    gpu_ctx.sync()
    eq((x, y, v), (hx, hy, hv))
    for d in (dx, dy, dv):
        gpu_ctx.device_free(d)
    pyr.close()


def test_select_small_chunks_ties_and_exhaustion(oracle):
    """The walk's rare paths: chunk capacity 64 (every histogram bin larger than a chunk -> the in-kernel radix sort),
    candidate ranges that run out (fallback gathers), massive exact ties (periodic image), fewer candidates than slots
    (KLT_NOT_FOUND fill, quirk Q6)."""
    from pyfeaturetrack_b200 import _capi, synth
    os.environ["KLT_B200_SELECT_CHUNK"] = "64"
    try:
        ctx = _capi.Context(_capi.default_ctx().device)
    finally:
        del os.environ["KLT_B200_SELECT_CHUNK"]
    try:
        kw = dict(nPyramidLevels=1, subsampling=2)
        tc = make_tc(**kw)
        p = oracle.Params(**kw)
        yy, xx = np.mgrid[0:240, 0:320]
        checker = (((xx // 8) + (yy // 8)) % 2 * 200 + 20).astype(np.uint8)            # exact ties everywhere
        sparse = np.full((240, 320), 90, np.uint8)
        sparse[100:110, 150:160] = 220                                                  # four corners: far fewer candidates than slots
        frames = [synth.frames(240, 320, [(0.0, 0.0)], seed=3)[0], checker, sparse]
        pyr = build_batch(ctx, tc, frames, _capi.PRECISION_STRICT)
        for n in (60, 700):
            x, y, v = batch_select(ctx, tc, pyr, n, False, _capi.SELECT_STRICT)
            for b, f in enumerate(frames):
                eq((x[b], y[b], v[b]), oracle_select_on_pyramid(oracle, p, f, n))
        assert (v[2] == -1).any() and (v[0] > 0).any()
        # replacement with small chunks: lose half
        x, y, v = batch_select(ctx, tc, pyr, 60, False, _capi.SELECT_STRICT)
        x2, y2, v2 = x.copy(), y.copy(), v.copy()
        x2[:, ::2] = -1.0; y2[:, ::2] = -1.0; v2[:, ::2] = -3
        gx, gy, gv = batch_select(ctx, tc, pyr, 60, True, _capi.SELECT_STRICT, x2, y2, v2)
        for b, f in enumerate(frames):
            eq((gx[b], gy[b], gv[b]), oracle_select_on_pyramid(oracle, p, f, 60, existing=(x2[b], y2[b], v2[b])))
        pyr.close()
    finally:
        ctx.close()


def test_dropin_select_and_replace_use_the_batch_chain(gpu_ctx, oracle):
    """KLTSelectGoodFeatures / KLTReplaceLostFeatures (drop-in API) on odd sizes and mindist variants == oracle."""
    from pyfeaturetrack_b200 import synth, selectGoodFeatures as sgf
    for (H, W, n, kw) in [(241, 323, 150, dict(mindist=3)), (200, 264, 64, dict(mindist=0)), (360, 488, 200, dict(mindist=25, min_eigenvalue=50))]:
        tc = make_tc(**kw)
        p = oracle.Params(**kw)
        f = synth.frames(H, W, [(0.0, 0.0)], seed=11)[0]
        fl = sgf.KLTSelectGoodFeatures(tc, f, n)
        want = oracle.select_good_features(p, f, n)
        got = (np.array([float(a.x) for a in fl]), np.array([float(a.y) for a in fl]), np.array([int(a.val) for a in fl]))
        eq(got, want)


def test_fractional_min_eigenvalue_and_sticky_assert_flag(gpu_ctx, oracle):
    """(1) tc.min_eigenvalue = k + 0.5 cuts where the reference's float comparison cuts (not at int(k + 0.5));
    (2) klt_track_features on DEVICE arrays without n_iterations does not wait: a window that leaves the image (the reference's
    AssertionError, trackFeaturesUtils.pyx:35) is reported by the next klt_sync."""
    from pyfeaturetrack_b200 import _capi, synth, selectGoodFeatures as sgf, trackFeatures as tf
    img = synth.frames(240, 320, [(0.0, 0.0)], seed=17)[0]
    x, y, v = oracle.select_good_features(oracle.Params(), img, 400)
    found = np.sort(v[v > 0])
    cut = float(found[len(found) // 2]) + 0.5
    tc = make_tc(min_eigenvalue=cut)
    fl = sgf.KLTSelectGoodFeatures(tc, img, 400)
    got = (np.array([float(a.x) for a in fl]), np.array([float(a.y) for a in fl]), np.array([int(a.val) for a in fl]))
    eq(got, oracle.select_good_features(oracle.Params(min_eigenvalue=cut), img, 400))
    assert (got[2] == -1).any()
    # sticky flag
    tc = make_tc()
    pyr = build_batch(gpu_ctx, tc, [img], _capi.PRECISION_FAST)
    n = 4
    hx, hy, hv = np.array([160.0, 2.0, 100.0, 50.0]), np.array([120.0, 2.0, 80.0, 60.0]), np.zeros(n, np.int32)    # feature 1 sits in the border
    dx, dy, dv = gpu_ctx.device_alloc(n * 8), gpu_ctx.device_alloc(n * 8), gpu_ctx.device_alloc(n * 4)
    gpu_ctx.memcpy(dx, hx, n * 8); gpu_ctx.memcpy(dy, hy, n * 8); gpu_ctx.memcpy(dv, hv, n * 4)
    params = sgf.make_params(tc)
    gpu_ctx.check(_capi.lib().klt_track_features(gpu_ctx.handle, C.byref(params), pyr.handle, pyr.handle, n, dx, dy, dv, None))
    with pytest.raises(AssertionError):
        gpu_ctx.sync()
    gpu_ctx.sync()                       # reported once
    for d in (dx, dy, dv):
        gpu_ctx.device_free(d)
    pyr.close()


@pytest.mark.parametrize("precision", ["windowed", "fast", "strict"])
def test_overlapped_device_pairs_equal_serial(gpu_ctx, oracle, precision):
    """klt_track_pairs_u8 with device-resident frames and lists (sub-batches tracked on a second stream while the next ones are
    built) gives exactly what the three separate calls give."""
    from pyfeaturetrack_b200 import _capi, synth, selectGoodFeatures as sgf, trackFeatures as tf
    prec = {"windowed": _capi.PRECISION_FAST_WINDOWED, "fast": _capi.PRECISION_FAST, "strict": _capi.PRECISION_STRICT}[precision]
    H, W, n, B = 240, 320, 120, 10
    tc = make_tc(nPyramidLevels=2, subsampling=2, max_residue=10.0)
    params, taps = sgf.make_params(tc), tf._taps_for_one_image(tc)
    pairs = [synth.frame_pair(H, W, seed=60 + i, shift=(1.0 + 0.3 * i, -2.0 + 0.4 * i)) for i in range(B)]
    f1 = np.ascontiguousarray(np.stack([p[0] for p in pairs])); f2 = np.ascontiguousarray(np.stack([p[1] for p in pairs]))
    sel = [oracle.select_good_features(oracle.Params(nPyramidLevels=2, subsampling=2), p[0], n) for p in pairs]
    x0 = np.stack([s[0] for s in sel]); y0 = np.stack([s[1] for s in sel]); v0 = np.stack([s[2] for s in sel]).astype(np.int32)
    ctx = gpu_ctx
    lib = _capi.lib()
    d1, d2 = ctx.device_alloc(f1.nbytes), ctx.device_alloc(f2.nbytes)
    dx, dy, dv = ctx.device_alloc(B * n * 8), ctx.device_alloc(B * n * 8), ctx.device_alloc(B * n * 4)
    ctx.memcpy(d1, f1, f1.nbytes); ctx.memcpy(d2, f2, f2.nbytes)
    p1, p2 = _capi.Pyramid(ctx, W, H, 2, 2, B), _capi.Pyramid(ctx, W, H, 2, 2, B)
    res = []
    for overlapped in (True, False):
        ctx.memcpy(dx, x0, B * n * 8); ctx.memcpy(dy, y0, B * n * 8); ctx.memcpy(dv, v0, B * n * 4)
        if overlapped:
            ctx.check(lib.klt_track_pairs_u8(ctx.handle, C.byref(params), C.byref(taps), prec, p1.handle, p2.handle, d1, d2, W, W * H, n, dx, dy, dv))
        else:
            ctx.check(lib.klt_pyr_build_u8(ctx.handle, p1.handle, d1, W, W * H, C.byref(taps), prec))
            ctx.check(lib.klt_pyr_build_u8(ctx.handle, p2.handle, d2, W, W * H, C.byref(taps), prec))
            ctx.check(lib.klt_track_features(ctx.handle, C.byref(params), p1.handle, p2.handle, n, dx, dy, dv, None))
        x, y, v = np.empty((B, n)), np.empty((B, n)), np.empty((B, n), np.int32)
        ctx.memcpy(x, dx, B * n * 8); ctx.memcpy(y, dy, B * n * 8); ctx.memcpy(v, dv, B * n * 4)
        ctx.sync()
        res.append((x, y, v))
    eq(res[0], res[1])
    assert (res[0][2] == 0).mean() > 0.8
    if precision == "strict":
        for b in range(B):
            want = oracle.track_features(oracle.Params(nPyramidLevels=2, subsampling=2, max_residue=10.0), pairs[b][0], pairs[b][1], *sel[b])[:3]
            eq((res[0][0][b], res[0][1][b], res[0][2][b]), want)
    for d in (d1, d2, dx, dy, dv):
        ctx.device_free(d)
    p1.close(); p2.close()


# ---- fused fast eigenvalue pass ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,kw", [((480, 640), dict(nPyramidLevels=2, subsampling=2)),
                                      ((243, 325), dict(nSkippedPixels=2)),
                                      ((300, 400), dict(window_width=15, window_height=15, nPyramidLevels=1, subsampling=2)),
                                      ((256, 384), dict(window_width=3, window_height=3, nPyramidLevels=1, subsampling=2))])
def test_fast_eigen_map_close_to_reference_map(gpu_ctx, oracle, shape, kw):
    """The fused pass (fp32, direct window sums) against the oracle's SAT-based map: the difference is bounded by the SAT's own
    float32 rounding (a few units on values of hundreds to thousands), i.e. tiny relative to the map's scale."""
    from pyfeaturetrack_b200 import _capi, synth, selectGoodFeatures as sgf
    tc = make_tc(**kw)
    p = oracle.Params(**kw)
    f = synth.frames(shape[0], shape[1], [(0.0, 0.0)], seed=21)[0]
    pyr = build_batch(gpu_ctx, tc, [f], _capi.PRECISION_FAST_WINDOWED)
    params = sgf.make_params(tc)
    nx, ny = C.c_int(), C.c_int()
    gpu_ctx.check(_capi.lib().klt_eigen_map_batch(gpu_ctx.handle, C.byref(params), pyr.handle, _capi.SELECT_FAST, None, C.byref(nx), C.byref(ny)))
    got = np.empty((ny.value, nx.value), np.float32)
    gpu_ctx.check(_capi.lib().klt_eigen_map_batch(gpu_ctx.handle, C.byref(params), pyr.handle, _capi.SELECT_FAST, got.ctypes.data, C.byref(nx), C.byref(ny)))
    _, gxs, gys = oracle.image_pyramids(p, f)
    hw = int(p.window_width / 2)
    bx = int(max(p.borderx, p.window_width / 2))
    want, _, _ = oracle.scan_good_features(gxs[0], gys[0], bx, bx, hw, hw, p.nSkippedPixels)
    assert got.shape == want.shape
    # exact window sums in float64 from the oracle's gradients: the fused pass must be much closer to these than the SAT map is
    exact, scale = _exact_eigen_map(p, gxs[0], gys[0])
    assert exact.shape == got.shape
    assert np.abs(got - exact).max() <= 2e-5 * scale
    assert np.abs(got - want).max() <= np.abs(want - exact).max() + 2e-5 * scale
    pyr.close()


def _exact_eigen_map(p, gx, gy):
    """float64 window sums + eigenvalue from the oracle's gradients, laid out like the scan's output."""
    hw = int(p.window_width / 2)
    bx = int(max(p.borderx, p.window_width / 2))
    gx, gy = gx.astype(np.float64), gy.astype(np.float64)

    def box(a):
        s = np.pad(a.cumsum(0).cumsum(1), ((1, 0), (1, 0)))
        k = 2 * hw + 1
        return s[k:, k:] - s[:-k, k:] - s[k:, :-k] + s[:-k, :-k]
    gxx, gxy, gyy = box(gx * gx), box(gx * gy), box(gy * gy)
    exact = 0.5 * ((gxx + gyy) - np.sqrt((gxx - gyy) ** 2 + 4 * gxy ** 2))
    step = p.nSkippedPixels + 1
    return exact[bx - hw:exact.shape[0] - (bx - hw):step, bx - hw:exact.shape[1] - (bx - hw):step], float((gxx + gyy).max())


@pytest.mark.parametrize("cfg", ["B", "C"])
def test_fast_selection_set_overlap(gpu_ctx, oracle, cfg):
    """select='fast' (fused pass on a fast image-only build) at configs B and C, as sets of selected pixels:
    * against the selection computed from EXACT (float64) window sums of the reference's gradients: >= 99.8 % -- the fused
      pass reproduces what exact arithmetic selects;
    * against the reference's own selection: what is left is the reference's float32 summed-area-table rounding (up to
      +-20 on eigenvalues of a few thousand at 1080p, several times that at 4K), which decides near-ties differently.  The
      fast mode must be as close to the reference as exact arithmetic is (measured on B200: 99.3-99.7 % at B, 97.0 % at C;
      SURVEY 7.3 expected 99.8-99.9 %)."""
    from pyfeaturetrack_b200 import synth, selectGoodFeatures as sgf, config
    H, W, n, L = (1080, 1920, 1000, 3) if cfg == "B" else (2160, 3840, 10000, 4)
    kw = dict(nPyramidLevels=L, subsampling=2)
    tc = make_tc(**kw)
    p = oracle.Params(**kw)
    f = synth.frames(H, W, [(0.0, 0.0)], seed=0)[0]
    config.set_precision(select="fast")
    fl = sgf.KLTSelectGoodFeatures(tc, f, n)
    got = {(int(a.x), int(a.y)) for a in fl if a.val > 0}
    sm = oracle.smooth(f.astype(np.float32), p.smooth_sigma(), p.cache)
    gx, gy = oracle.gradients(sm, p.grad_sigma, p.cache)
    rx, ry, rv, _ = oracle.select_from_gradients(p, gx, gy, n)
    ref = {(int(a), int(b)) for a, b, c in zip(rx, ry, rv) if c > 0}
    exact_map, _ = _exact_eigen_map(p, gx, gy)
    ex, ey, ev = oracle.select_from_map(p, exact_map, W, H, n)
    exact = {(int(a), int(b)) for a, b, c in zip(ex, ey, ev) if c > 0}
    assert len(got) == len(ref) == len(exact) == n

    def ov(a, b):
        return len(a & b) / float(n)
    print("set overlap fast/exact %.4f  fast/reference %.4f  exact/reference %.4f" % (ov(got, exact), ov(got, ref), ov(exact, ref)))
    assert ov(got, exact) >= 0.998
    assert ov(got, ref) >= ov(exact, ref) - 0.003
    assert ov(got, ref) >= (0.99 if cfg == "B" else 0.96)


# ---- sequences -----------------------------------------------------------------------------------------------------------------
def _sequence_frames(H, W, nframes, nseq, speed):
    from pyfeaturetrack_b200 import synth
    shifts = [(s[0] * speed, s[1] * speed) for s in synth.sequence_shifts(nframes)]
    return [synth.frames(H, W, shifts, seed=100 + s) for s in range(nseq)]        # [sequence][frame]


def _oracle_sequence(oracle, p, frames, n, replace=True):
    """The reference flow for one sequence: select, then per frame KLTTrackFeatures (sequentialMode) + replacement on
    pyramid_last's level-0 gradients.  Returns the lists after every frame and the status codes after tracking."""
    state = {}
    pyr0 = oracle.image_pyramids(p, frames[0])
    x, y, v, _ = oracle.select_from_gradients(p, pyr0[1][0], pyr0[2][0], n)
    state["pyramid_last"] = pyr0
    out = [(x.copy(), y.copy(), v.copy(), None)]
    for k in range(1, len(frames)):
        x, y, v, _ = oracle.track_features(p, frames[k - 1], frames[k], x, y, v, state)
        vt = v.copy()
        if replace:
            _, gxs, gys = state["pyramid_last"]
            x, y, v, _ = oracle.select_from_gradients(p, gxs[0], gys[0], n, existing=(x, y, v))
        out.append((x.copy(), y.copy(), v.copy(), vt))
    return out


def _run_sequence(ctx, tc, seqs, n, precision, select_mode, replace=True, taps=None):
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf, trackFeatures as tf
    B, nfr = len(seqs), len(seqs[0])
    H, W = seqs[0][0].shape
    taps = tf._taps_for_one_image(tc) if taps is None else taps
    q = _capi.Sequence(ctx, sgf.make_params(tc), taps, W, H, B, n, precision, select_mode)
    q.start(np.ascontiguousarray(np.stack([s[0] for s in seqs])))
    out = [q.features()]
    for k in range(1, nfr):
        q.step(np.ascontiguousarray(np.stack([s[k] for s in seqs])), replace=replace)
        out.append(q.features())
    q.sync()
    graph = q.uses_graph()
    q.close()
    return out, graph


def test_sequence_strict_equals_oracle_20_frames_4_sequences(gpu_ctx, oracle):
    """BASELINE config D, shortened and reduced in size: 4 lock-stepped sequences x 21 frames, per-frame replacement, STRICT
    pyramids + STRICT selection: every feature list after every frame (positions, status codes after tracking, replacement
    slots and values) == the oracle's, which equals the reference's."""
    from pyfeaturetrack_b200 import _capi
    kw = dict(nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    tc = make_tc(**kw)
    p = oracle.Params(**kw)
    n, nfr, nseq = 300, 21, 4
    seqs = _sequence_frames(480, 640, nfr, nseq, speed=5.0)
    got, graph = _run_sequence(gpu_ctx, tc, seqs, n, _capi.PRECISION_STRICT, _capi.SELECT_STRICT)
    assert graph, "steps were not replayed from a CUDA graph"
    lost = 0
    for s in range(nseq):
        want = _oracle_sequence(oracle, p, seqs[s], n)
        for k in range(nfr):
            gx, gy, gv, gvt = got[k]
            eq((gx[s], gy[s], gv[s]), want[k][:3])
            if k:
                assert np.array_equal(gvt[s], want[k][3])
                lost += int((want[k][3] < 0).sum())
    assert lost > 20 * nseq          # the test must exercise replacement


def test_sequence_1080p_strict_and_graph_vs_plain(gpu_ctx, oracle):
    """Full-size config D frames (1080p, 1000 features), 2 sequences x 4 frames: == oracle; and the CUDA-graph replay gives
    exactly what plain launches give."""
    from pyfeaturetrack_b200 import _capi
    kw = dict(nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    tc = make_tc(**kw)
    p = oracle.Params(**kw)
    n, nfr, nseq = 1000, 5, 2
    seqs = _sequence_frames(1080, 1920, nfr, nseq, speed=6.0)
    got, graph = _run_sequence(gpu_ctx, tc, seqs, n, _capi.PRECISION_STRICT, _capi.SELECT_STRICT)
    assert graph
    want = _oracle_sequence(oracle, p, seqs[0], n)
    for k in range(nfr):
        eq((got[k][0][0], got[k][1][0], got[k][2][0]), want[k][:3])
    os.environ["KLT_B200_NO_GRAPH"] = "1"
    try:
        plain, graph2 = _run_sequence(gpu_ctx, tc, seqs, n, _capi.PRECISION_STRICT, _capi.SELECT_STRICT)
    finally:
        del os.environ["KLT_B200_NO_GRAPH"]
    assert not graph2
    for k in range(nfr):
        for a, b in zip(got[k], plain[k]):
            assert np.array_equal(a, b)


def test_sequence_fast_modes_track_the_strict_sequence(gpu_ctx, oracle):
    """Windowed tracking + fused fast selection over 50 frames without replacement feedback differences: tracking agrees with
    the oracle's statuses on >= 99.9 % of the features and within 1e-3 px per frame when both start each frame from the same
    list (per-frame comparison, lists re-synchronised from the oracle), and the free-running fast sequence keeps as many
    features alive as the strict one (+-1 %)."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf, trackFeatures as tf
    kw = dict(nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    tc = make_tc(**kw)
    p = oracle.Params(**kw)
    n, nfr = 400, 51
    seqs = _sequence_frames(480, 640, nfr, 2, speed=3.0)
    want = [_oracle_sequence(oracle, p, s, n) for s in seqs]
    H, W = seqs[0][0].shape
    for precision in (_capi.PRECISION_FAST, _capi.PRECISION_FAST_WINDOWED):
        q = _capi.Sequence(gpu_ctx, sgf.make_params(tc), tf._taps_for_one_image(tc), W, H, 2, n, precision, _capi.SELECT_STRICT)
        q.start(np.ascontiguousarray(np.stack([s[0] for s in seqs])), select=False)
        match = tot = 0
        worst = 0.0
        for k in range(1, nfr):
            prev = [want[s][k - 1] for s in range(2)]
            q.set_features(np.stack([a[0] for a in prev]), np.stack([a[1] for a in prev]), np.stack([a[2] for a in prev]))
            q.step(np.ascontiguousarray(np.stack([s[k] for s in seqs])), replace=False)
            gx, gy, gv, gvt = q.features()
            for s in range(2):
                wx, wy, _, wvt = want[s][k]
                # the oracle's list after replacement differs from the tracked one only in the replaced slots
                live = prev[s][2] >= 0
                match += int((gvt[s][live] == wvt[live]).sum()); tot += int(live.sum())
                both = live & (gvt[s] == 0) & (wvt == 0)
                if both.any():
                    worst = max(worst, float(np.abs(gx[s][both] - wx[both]).max()), float(np.abs(gy[s][both] - wy[both]).max()))
        q.sync()
        q.close()
        assert match / float(tot) >= 0.999, "status match %.5f" % (match / float(tot))
        assert worst <= 1e-3, "max position error %g px" % worst
    # free-running fast sequence (windowed tracking + fused fast selection)
    got, _ = _run_sequence(gpu_ctx, tc, seqs, n, _capi.PRECISION_FAST_WINDOWED, _capi.SELECT_FAST)
    for s in range(2):
        alive_fast = np.mean([(got[k][3][s] == 0).sum() for k in range(1, nfr)])
        alive_ref = np.mean([(want[s][k][3] == 0).sum() for k in range(1, nfr)])
        assert abs(alive_fast - alive_ref) <= 0.01 * n, (alive_fast, alive_ref)
        assert (got[-1][2][s] >= 0).all()


# ---- the reference's own outputs at BASELINE's sizes (tests/golden/reference_golden_fullsize.npz) ------------------------------
def test_fullsize_goldens_config_B_and_C(gpu_ctx, golden_fullsize):
    """Drop-in API, STRICT: selection and tracking at 1080p / 1000 features and 4K / 10 000 features == the arrays the unmodified
    reference produced (positions, values and status codes compared with ==)."""
    from pyfeaturetrack_b200 import synth, selectGoodFeatures as sgf, trackFeatures as tf, config
    config.set_precision(track="strict", select="strict")
    for (H, W, n, L, key) in ((1080, 1920, 1000, 3, "B"), (2160, 3840, 10000, 4, "C")):
        imgs = synth.frame_pair(H, W, seed=0)
        tc = make_tc(nPyramidLevels=L, subsampling=2, max_residue=10.0)
        fl = sgf.KLTSelectGoodFeatures(tc, imgs[0], n)
        got = (np.array([float(a.x) for a in fl]), np.array([float(a.y) for a in fl]), np.array([int(a.val) for a in fl]))
        eq(got, golden_fullsize["%s_sel%d" % (key, n)])
        tf.KLTTrackFeatures(tc, imgs[0], imgs[1], fl)
        got = (np.array([float(a.x) for a in fl]), np.array([float(a.y) for a in fl]), np.array([int(a.val) for a in fl]))
        eq(got, golden_fullsize["%s_trk%d" % (key, n)])


def test_fullsize_golden_config_D_sequence(gpu_ctx, golden_fullsize):
    """klt_sequence, STRICT + STRICT, on the 1080p sequence of the golden file: after every frame the lists equal the
    reference's (tracking result = val_tracked + positions of the tracked features; after replacement = x, y, val)."""
    from pyfeaturetrack_b200 import _capi, synth
    g = golden_fullsize["D_seq1000"]
    nfr = 5
    shifts = [(s[0] * 6, s[1] * 6) for s in synth.sequence_shifts(nfr)]
    frames = synth.frames(1080, 1920, shifts, seed=101)
    tc = make_tc(nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    got, _ = _run_sequence(gpu_ctx, tc, [frames, frames], 1000, _capi.PRECISION_STRICT, _capi.SELECT_STRICT)
    for s in range(2):
        eq((got[0][0][s], got[0][1][s], got[0][2][s]), g[0])
        for k in range(1, nfr):
            assert np.array_equal(got[k][3][s], g[2 * k - 1][2].astype(np.int32))          # status codes after tracking
            eq((got[k][0][s], got[k][1][s], got[k][2][s]), g[2 * k])                        # lists after replacement


def test_sequence_fast_select_outside_the_fused_pass_equals_strict(gpu_ctx):
    """The fused eigenvalue pass needs a symmetric 7-tap gradient smoother.  With one outer tap 1e-6 relative off it declines,
    and a KLT_SELECT_FAST sequence must take the table-based pass instead, with its own summed-area-table workspace, on plain
    launches and in graph replay: every list of every step equals the KLT_SELECT_STRICT run on the same taps and frames."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf, trackFeatures as tf
    kw = dict(nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    tc = make_tc(**kw)
    seqs = _sequence_frames(360, 480, 10, 3, speed=4.0)
    H, W = seqs[0][0].shape
    taps = tf._taps_for_one_image(tc)
    assert taps.grad_gauss.n == 7
    params = sgf.make_params(tc)
    pyr = _capi.Pyramid(gpu_ctx, W, H, 3, 2, 1)
    val = np.empty(H * W, np.float32)
    nx, ny = C.c_int(), C.c_int()
    codes = []
    for perturb in (False, True):
        if perturb:
            taps.grad_gauss.taps[0] *= 1 + 1e-6
        pyr.build_u8(np.ascontiguousarray(seqs[0][0]), taps, _capi.PRECISION_FAST_WINDOWED)
        codes.append(_capi.lib().klt_eigen_map_batch(gpu_ctx.handle, C.byref(params), pyr.handle, _capi.SELECT_FAST,
                                                     val.ctypes.data, C.byref(nx), C.byref(ny)))
    pyr.close()
    assert codes == [0, _capi.KLT_ERR_UNSUPPORTED]
    runs = {}
    for sel in (_capi.SELECT_FAST, _capi.SELECT_STRICT):
        runs[sel], graph = _run_sequence(gpu_ctx, tc, seqs, 200, _capi.PRECISION_FAST_WINDOWED, sel, taps=taps)
        assert graph
    assert sum(int((o[3] != 0).sum()) for o in runs[_capi.SELECT_STRICT][1:]) > 0, "nothing was replaced"
    for k, (got, want) in enumerate(zip(runs[_capi.SELECT_FAST], runs[_capi.SELECT_STRICT])):
        for a, b in zip(got, want):
            assert np.array_equal(a, b), k


@pytest.mark.gpu
@pytest.mark.parametrize("precision,select,levels", [pytest.param("windowed", "fast", 3, id="windowed-fast"),
                                                     pytest.param("fast", "strict", 3, id="fast-strict"),
                                                     pytest.param("strict", "strict", 3, id="strict-strict"),
                                                     pytest.param("windowed", "strict", 1, id="windowed-strict-one-level")])
def test_sequence_second_stream_changes_nothing(gpu_ctx, monkeypatch, precision, select, levels):
    """The eigenvalue pass of a step runs on the context's second stream beside the decimations and the tracking kernel
    ($KLT_B200_SEQ_OVERLAP, on by default): every list of every frame must equal the single-stream run bit for bit, replayed
    from the graph and with plain launches.  A profiled run (plain launches, one stream) shows the tracker the pyramids'
    precision selects; with one level, the level-0 gradient planes the table-based selection builds must not move an
    image-only pyramid off the windowed tracker."""
    from pyfeaturetrack_b200 import _capi
    kw = dict(nPyramidLevels=levels, subsampling=2, max_residue=10.0, sequentialMode=True)
    tc = make_tc(**kw)
    seqs = _sequence_frames(360, 480, 9, 3, speed=4.0)
    prec = dict(windowed=_capi.PRECISION_FAST_WINDOWED, fast=_capi.PRECISION_FAST, strict=_capi.PRECISION_STRICT)[precision]
    sel = _capi.SELECT_FAST if select == "fast" else _capi.SELECT_STRICT
    runs = {}
    for overlap in ("1", "0"):
        for graph in (True, False):
            monkeypatch.setenv("KLT_B200_SEQ_OVERLAP", overlap)
            if graph:
                monkeypatch.delenv("KLT_B200_NO_GRAPH", raising=False)
            else:
                monkeypatch.setenv("KLT_B200_NO_GRAPH", "1")
            runs[(overlap, graph)], used = _run_sequence(gpu_ctx, tc, seqs, 200, prec, sel)
            assert used == graph
    gpu_ctx.profile(True)
    gpu_ctx.profile_reset()
    try:
        runs["profiled"], _ = _run_sequence(gpu_ctx, tc, seqs, 200, prec, sel)
        kernels = gpu_ctx.profile_read()
    finally:
        gpu_ctx.profile(False)
    tracker = dict(windowed="lk_windowed", fast="lk_track_rows", strict="lk_track")[precision]
    assert [k for k in ("lk_windowed", "lk_track_rows", "lk_track") if k in kernels] == [tracker], sorted(kernels)
    assert kernels[tracker]["launches"] == len(seqs[0]) - 1
    ref = runs[("0", False)]
    for key, got in runs.items():
        for k in range(len(ref)):
            for a, b in zip(got[k], ref[k]):
                assert np.array_equal(a, b), (key, k)


@pytest.mark.parametrize("precision,select,shape,B", [("windowed", "fast", (1080, 1920), 8), ("windowed", "strict", (1080, 1920), 8),
                                                       ("strict", "strict", (480, 640), 4), ("fast", "strict", (480, 640), 4)])
def test_sequence_run_ahead_equals_step_by_step(gpu_ctx, monkeypatch, precision, select, shape, B):
    """The front half of step k + 1 (build, eigenvalue maps) overlaps the back half of step k (tracking, replacement) only when
    the host does not wait between steps.  24 steps enqueued back to back -- device-resident frames, results copied into one
    pinned set per step, one synchronisation at the end -- must equal the same run with a synchronisation after every step and
    the single-stream run, list by list."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf, trackFeatures as tf
    kw = dict(nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    tc = make_tc(**kw)
    H, W = shape
    n, nfr = 500, 25
    seqs = _sequence_frames(H, W, nfr, 2, speed=4.0)
    frames = np.ascontiguousarray(np.stack([np.stack([seqs[s % 2][(k + s // 2) % nfr] for s in range(B)]) for k in range(nfr)]))
    prec = dict(windowed=_capi.PRECISION_FAST_WINDOWED, fast=_capi.PRECISION_FAST, strict=_capi.PRECISION_STRICT)[precision]
    sel = _capi.SELECT_FAST if select == "fast" else _capi.SELECT_STRICT
    dfr = gpu_ctx.device_alloc(frames.nbytes)
    gpu_ctx.memcpy(dfr, frames, frames.nbytes)
    gpu_ctx.sync()
    per = B * H * W
    runs = {}
    try:
        for mode in ("run_ahead", "stepwise", "one_stream"):
            monkeypatch.setenv("KLT_B200_SEQ_OVERLAP", "0" if mode == "one_stream" else "1")
            q = _capi.Sequence(gpu_ctx, sgf.make_params(tc), tf._taps_for_one_image(tc), W, H, B, n, prec, sel)
            outs = [(gpu_ctx.pinned_array((B, n), np.float64), gpu_ctx.pinned_array((B, n), np.float64),
                     gpu_ctx.pinned_array((B, n), np.int32), gpu_ctx.pinned_array((B, n), np.int32)) for _ in range(nfr - 1)]
            q.start(dfr)
            for k in range(1, nfr):
                q.step(dfr + k * per, out=outs[k - 1])
                if mode == "stepwise":
                    q.sync()
            q.sync()
            assert q.uses_graph()
            runs[mode] = [tuple(np.array(a) for a in o) for o in outs]
            q.close()
            for o in outs:
                for a in o:
                    gpu_ctx.free_pinned(a)
    finally:
        gpu_ctx.device_free(dfr)
    lost = sum(int((o[3] != 0).sum()) for o in runs["one_stream"])
    assert lost > 0, "the scenario loses no feature: nothing would be replaced"
    for mode in ("run_ahead", "stepwise"):
        for k, (got, want) in enumerate(zip(runs[mode], runs["one_stream"])):
            for a, b in zip(got, want):
                assert np.array_equal(a, b), (mode, k)
