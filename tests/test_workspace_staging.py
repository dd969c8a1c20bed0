"""Host and device arguments of the C ABI and the context workspace they are staged through.

Every entry point that takes "host or device" arrays must give the same results (==) for either kind, a context whose
workspace grows and shrinks between calls must give what a fresh context gives, and the tracking status words (iteration
count, assert word) must reach the caller the same way from klt_track_features and from klt_sequence."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W, H = 320, 240


@pytest.fixture(scope="module")
def ctx():
    from pyfeaturetrack_b200 import _capi
    c = _capi.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def frames():
    from pyfeaturetrack_b200 import synth
    return synth.frame_pair(H, W, seed=7)


def make_tc(**kw):
    from pyfeaturetrack_b200 import klt, selectGoodFeatures, trackFeatures
    selectGoodFeatures.KLT_verbose = 0
    trackFeatures.KLT_verbose = 0
    tc = klt.KLT_TrackingContext()
    for k, v in kw.items():
        setattr(tc, k, v)
    tc.KLTUpdateTCBorder()
    return tc


class Args:
    """Arguments of one call: numpy arrays passed as they are (host) or copied to klt_device_alloc buffers (device)."""

    def __init__(self, ctx, device):
        self.ctx, self.device, self.bufs, self.outs = ctx, device, [], []

    def arg(self, a, device=None):
        if not (self.device if device is None else device):
            return a.ctypes.data
        p = self.ctx.device_alloc(max(a.nbytes, 1))
        self.ctx.memcpy(p, a, a.nbytes)
        self.bufs.append(p)
        self.outs.append((a, p))
        return p

    def results(self):
        """Copies every device buffer back into its array and frees it."""
        for a, p in self.outs:
            self.ctx.memcpy(a, p, a.nbytes)
        self.ctx.sync()
        for p in self.bufs:
            self.ctx.device_free(p)
        self.bufs, self.outs = [], []


def kernels(tc):
    from pyfeaturetrack_b200 import _capi, convolve
    g, _ = convolve._kernels_for_smoothing(1.5)
    gg, gd = convolve._kernels_for_gradients(tc.grad_sigma)
    return _capi.Kernel1D.from_taps(g), _capi.Kernel1D.from_taps(gg), _capi.Kernel1D.from_taps(gd)


def pyramids(ctx, tc, frames, precision):
    from pyfeaturetrack_b200 import _capi, trackFeatures as tf
    out = []
    for f in frames:
        p = _capi.Pyramid(ctx, f.shape[1], f.shape[0], int(tc.nPyramidLevels), int(tc.subsampling), 1)
        p.build_u8(np.ascontiguousarray(f), tf._taps_for_one_image(tc), precision)
        out.append(p)
    return out


def select(ctx, tc, pyr, n):
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf
    x, y, v = np.zeros(n), np.zeros(n), np.zeros(n, np.int32)
    ctx.check(_capi.lib().klt_select_good_features_batch(ctx.handle, C.byref(sgf.make_params(tc)), pyr.handle, n, 0,
                                                         _capi.SELECT_STRICT, x.ctypes.data, y.ctypes.data, v.ctypes.data))
    return x, y, v


# ---- one call per entry point, host (device=False) or device (device=True) arrays; mixed: inputs of the other kind ------
def call_convolve(ctx, frames, device, mixed=False, scale=1):
    from pyfeaturetrack_b200 import _capi
    lib = _capi.lib()
    img = np.ascontiguousarray(np.tile(frames[0], (scale, scale)), np.float32)
    out = np.zeros_like(img)
    g, _, _ = kernels(make_tc())
    a = Args(ctx, device)
    ctx.check(lib.klt_convolve_separable_f32(ctx.handle, a.arg(img, device != mixed), img.shape[1], img.shape[0], C.byref(g),
                                            C.byref(g), _capi.PRECISION_STRICT, a.arg(out)))
    a.results()
    return (out,)


def call_gradients(ctx, frames, device, mixed=False, scale=1):
    from pyfeaturetrack_b200 import _capi
    lib = _capi.lib()
    img = np.ascontiguousarray(np.tile(frames[1], (scale, scale)), np.float32)
    gx, gy = np.zeros_like(img), np.zeros_like(img)
    _, gg, gd = kernels(make_tc())
    a = Args(ctx, device)
    ctx.check(lib.klt_gradients_f32(ctx.handle, a.arg(img, device != mixed), img.shape[1], img.shape[0], C.byref(gg), C.byref(gd),
                                    _capi.PRECISION_STRICT, a.arg(gx), a.arg(gy)))
    a.results()
    return gx, gy


def call_scan(ctx, frames, device, mixed=False, scale=1):
    from pyfeaturetrack_b200 import _capi
    lib = _capi.lib()
    gx, gy = call_gradients(ctx, frames, False, scale=scale)
    h, w = gx.shape
    b, hw, skip = 4, 3, 1
    nx, ny = (w - 2 * b + skip) // (skip + 1), (h - 2 * b + skip) // (skip + 1)
    val = np.zeros((ny, nx), np.float32)
    a = Args(ctx, device)
    ctx.check(lib.klt_scan_good_features(ctx.handle, a.arg(gx, device != mixed), a.arg(gy, device != mixed), w, h, b, b, hw, hw,
                                         skip, a.arg(val)))
    a.results()
    return (val,)


def call_extract_patch(ctx, frames, device, mixed=False, scale=1):
    from pyfeaturetrack_b200 import _capi
    lib = _capi.lib()
    img = np.ascontiguousarray(np.tile(frames[0], (scale, scale)), np.float32)
    out = np.zeros((7, 9), np.float32)
    a = Args(ctx, device)
    ctx.check(lib.klt_extract_patch(ctx.handle, a.arg(img, device != mixed), img.shape[1], img.shape[0], 100.3, 57.8, 7, 9,
                                    a.arg(out)))
    a.results()
    return (out,)


def call_track_iterate(ctx, frames, device, mixed=False, scale=1):
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf
    lib = _capi.lib()
    tc = make_tc()
    params = sgf.make_params(tc)
    img1 = np.ascontiguousarray(frames[0], np.float32)
    img2 = np.ascontiguousarray(frames[1], np.float32)
    gx2, gy2 = call_gradients(ctx, frames, False)
    n = int(tc.window_width)
    gx1, gy1 = call_gradients(ctx, (frames[1], frames[0]), False)
    patches = [np.ascontiguousarray(im[100:100 + n, 150:150 + n]) for im in (img1, gx1, gy1)]
    x2, y2 = C.c_float(), C.c_float()
    st, it = C.c_int32(), C.c_int32()
    a = Args(ctx, device)
    ctx.check(lib.klt_track_iterate(ctx.handle, C.byref(params), 153.0, 103.0, a.arg(patches[1], device != mixed),
                                    a.arg(patches[2], device != mixed), a.arg(patches[0], device != mixed), a.arg(img2), a.arg(gx2),
                                    a.arg(gy2), W, H, C.byref(x2), C.byref(y2), C.byref(st), C.byref(it)))
    a.results()
    return np.array([x2.value, y2.value, st.value, it.value]),


def call_patch_combine(ctx, frames, device, mixed=False, scale=1):
    from pyfeaturetrack_b200 import _capi
    lib = _capi.lib()
    img2 = np.ascontiguousarray(np.tile(frames[1], (scale, scale)), np.float32)
    p1 = np.ascontiguousarray(frames[0][50:57, 60:69], np.float32)
    outs = []
    for mode in (0, 1):
        out = np.zeros_like(p1)
        a = Args(ctx, device)
        ctx.check(lib.klt_patch_combine(ctx.handle, a.arg(p1, device != mixed), a.arg(img2, device != mixed), img2.shape[1],
                                        img2.shape[0], 64.2, 53.9, 7, 9, mode, a.arg(out)))
        a.results()
        outs.append(out)
    return tuple(outs)


def call_eigen_map(ctx, frames, device, mixed=False, scale=1):
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf
    lib = _capi.lib()
    tc = make_tc()
    params = sgf.make_params(tc)
    outs = []
    for precision, mode in ((_capi.PRECISION_STRICT, _capi.SELECT_STRICT), (_capi.PRECISION_FAST_WINDOWED, _capi.SELECT_FAST)):
        (pyr,) = pyramids(ctx, tc, [np.tile(frames[0], (scale, scale))], precision)
        nx, ny = C.c_int(), C.c_int()
        ctx.check(lib.klt_eigen_map_batch(ctx.handle, C.byref(params), pyr.handle, mode, None, C.byref(nx), C.byref(ny)))
        val = np.zeros((ny.value, nx.value), np.float32)
        a = Args(ctx, device)
        ctx.check(lib.klt_eigen_map_batch(ctx.handle, C.byref(params), pyr.handle, mode, a.arg(val), C.byref(nx), C.byref(ny)))
        a.results()
        outs.append(val)
        pyr.close()
    return tuple(outs)


def call_select(ctx, frames, device, mixed=False, scale=1):
    """SELECTING_ALL, then REPLACING_SOME after knocking out every third feature; unmasked, then with a mask that is host or
    device (mixed: the other kind than the feature arrays)."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf
    lib = _capi.lib()
    tc = make_tc(mindist=5)
    params = sgf.make_params(tc)
    img = np.tile(frames[0], (scale, scale))
    (pyr,) = pyramids(ctx, tc, [img], _capi.PRECISION_STRICT)
    mask = np.ones(img.shape, np.uint8)
    mask[:, : img.shape[1] // 3] = 0
    n = 300
    outs = []
    for masked in (False, True):
        x, y, v = np.zeros(n), np.zeros(n), np.zeros(n, np.int32)
        for replace in (0, 1):
            if replace:
                v[::3] = -1
            a = Args(ctx, device)
            px, py, pv = a.arg(x), a.arg(y), a.arg(v)
            if masked:
                ctx.check(lib.klt_select_good_features_batch_masked(ctx.handle, C.byref(params), pyr.handle, n, replace,
                                                                    _capi.SELECT_STRICT, a.arg(mask, device != mixed),
                                                                    img.shape[1], 0, px, py, pv))
            else:
                ctx.check(lib.klt_select_good_features_batch(ctx.handle, C.byref(params), pyr.handle, n, replace,
                                                             _capi.SELECT_STRICT, px, py, pv))
            a.results()
            outs += [x.copy(), y.copy(), v.copy()]
    pyr.close()
    return tuple(outs)


def call_track(ctx, frames, device, mixed=False, scale=1, kind="plain"):
    """klt_track_features / _fb (with and without fb_error) / _affine on features selected on frame 1, with n_iterations."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf
    lib = _capi.lib()
    kw = dict(affineConsistencyCheck=1, max_residue=10.0) if kind == "affine" else {}
    tc = make_tc(**kw)
    params = sgf.make_params(tc)
    fr = [np.tile(f, (scale, scale)) for f in frames]
    pyr1, pyr2 = pyramids(ctx, tc, fr, _capi.PRECISION_STRICT)
    x, y, v = select(ctx, tc, pyr1, 200 * scale)
    n = x.size
    fb = np.full(n, 7.0, np.float32)
    it = C.c_int64()
    a = Args(ctx, device)
    px, py, pv = a.arg(x), a.arg(y), a.arg(v)
    if kind == "plain":
        ctx.check(lib.klt_track_features(ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, n, px, py, pv, C.byref(it)))
    elif kind in ("fb", "fb_no_error"):
        ctx.check(lib.klt_track_features_fb(ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, n, 0.5, px, py, pv,
                                            a.arg(fb, device != mixed) if kind == "fb" else None, C.byref(it)))
    else:
        aff = _capi.AffineState(ctx, n, int(tc.affine_window_width), int(tc.affine_window_height))
        ctx.check(lib.klt_track_features_affine(ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, n, px, py, pv, aff.handle,
                                                C.byref(it)))
        has, ax, ay, A = aff.download()
        aff.close()
    a.results()
    pyr1.close(); pyr2.close()
    out = (x, y, v, np.array([it.value]))
    if kind == "fb":
        out += (fb,)
    if kind == "affine":
        out += (has, ax, ay, A)
    return out


CALLS = dict(convolve=call_convolve, gradients=call_gradients, scan=call_scan, extract_patch=call_extract_patch,
             track_iterate=call_track_iterate, patch_combine=call_patch_combine, eigen_map=call_eigen_map, select=call_select,
             track=call_track, track_fb=lambda *a, **k: call_track(*a, kind="fb", **k),
             track_fb_no_error=lambda *a, **k: call_track(*a, kind="fb_no_error", **k),
             track_affine=lambda *a, **k: call_track(*a, kind="affine", **k))


def assert_same(got, want, what):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        assert np.array_equal(g, w), (what, i)


@pytest.mark.parametrize("name", sorted(CALLS))
def test_host_and_device_arguments_give_identical_results(ctx, frames, name):
    host = CALLS[name](ctx, frames, False)
    assert_same(CALLS[name](ctx, frames, True), host, (name, "device"))
    assert_same(CALLS[name](ctx, frames, True, mixed=True), host, (name, "device outputs, host inputs"))
    assert_same(CALLS[name](ctx, frames, False, mixed=True), host, (name, "host outputs, device inputs"))


def test_workspace_growth_between_calls(frames):
    """Small, large and small calls of different entry points on one context (its workspace grows, and a grown workspace
    serves the smaller calls) give what a fresh context gives for each call."""
    from pyfeaturetrack_b200 import _capi
    plan = [("convolve", 1), ("track", 3), ("convolve", 1), ("select", 3), ("scan", 1), ("track_fb", 1), ("gradients", 3),
            ("extract_patch", 1), ("track_affine", 2), ("patch_combine", 1), ("eigen_map", 3), ("track", 1)]
    shared = _capi.Context(0)
    try:
        for name, scale in plan:
            for device in (False, True):
                got = CALLS[name](shared, frames, device, scale=scale)
                fresh = _capi.Context(0)
                try:
                    want = CALLS[name](fresh, frames, device, scale=scale)
                finally:
                    fresh.close()
                assert_same(got, want, (name, scale, device))
    finally:
        shared.close()


def test_iterations_of_a_track_equal_those_of_a_one_step_sequence(ctx, frames):
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf, trackFeatures as tf
    tc = make_tc()
    params = sgf.make_params(tc)
    for precision in (_capi.PRECISION_STRICT, _capi.PRECISION_FAST, _capi.PRECISION_FAST_WINDOWED):
        pyr1, pyr2 = pyramids(ctx, tc, frames, precision)
        x, y, v = select(ctx, tc, pyr1, 300)
        seq = _capi.Sequence(ctx, params, tf._taps_for_one_image(tc), W, H, 1, x.size, precision, _capi.SELECT_STRICT)
        seq.start(np.ascontiguousarray(frames[0][None]), select=False)
        seq.set_features(x[None], y[None], v[None])
        it = C.c_int64()
        ctx.check(_capi.lib().klt_track_features(ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, x.size, x.ctypes.data,
                                                 y.ctypes.data, v.ctypes.data, C.byref(it)))
        seq.step(np.ascontiguousarray(frames[1][None]), replace=False)
        assert seq.sync() == it.value > 0, precision
        sx, sy, sv, _ = seq.features()
        assert np.array_equal(sx[0], x) and np.array_equal(sy[0], y) and np.array_equal(sv[0], v), precision
        seq.close(); pyr1.close(); pyr2.close()


def test_window_leaving_the_image_raises_now_or_at_sync(ctx):
    """Host arrays raise KLT_ERR_ASSERT from the call; device arrays without n_iterations raise it from klt_sync."""
    from pyfeaturetrack_b200 import _capi, synth, selectGoodFeatures as sgf
    f1, f2 = synth.frames(240, 320, [(0.0, 0.0), (0.0, -15.0)], seed=0)
    tc = make_tc(nPyramidLevels=3, subsampling=2)
    params = sgf.make_params(tc)
    pyr2, pyr1 = pyramids(ctx, tc, [f1, f2], _capi.PRECISION_STRICT)
    x, y, v = np.full(4, 5.0), np.array([60.0, 100.0, 140.0, 180.0]), np.zeros(4, np.int32)   # level 2 starts at x = 1.25
    track = _capi.lib().klt_track_features
    with pytest.raises(AssertionError):
        ctx.check(track(ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, 4, x.ctypes.data, y.ctypes.data, v.ctypes.data, None))
    a = Args(ctx, True)
    ctx.check(track(ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, 4, a.arg(x), a.arg(y), a.arg(v), None))
    with pytest.raises(AssertionError):
        ctx.sync()
    a.results()
    ctx.sync()                       # the flag is cleared once reported
    pyr1.close(); pyr2.close()
