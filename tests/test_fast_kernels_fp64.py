"""The FAST and FAST_WINDOWED pyramid kernels and the fused eigenvalue pass against a float64 reference.

The reference does not round: plain NumPy float64 separable convolutions with SciPy's 'reflect' border, fed with the taps
of the klt_taps struct the GPU receives.  Every GPU image must lie within an error bound derived from the fp32 arithmetic
the kernels do.  For one separable pass with taps h (n_h of them) and v (n_v), input error e_in and M = max|input|:

    e_out <= A * e_in + (n_h + n_v + 4) * u * A * M,    A = sum|h| * sum|v|,  u = 2**-24

n_h + n_v counts the roundings of the two FMA chains; the 4 covers the rounding of the taps to float (one per 1-D pass),
the intermediate between the two passes and the store.  The bound is applied stage by stage: level 0 from the exact frame;
level l from level l - 1 twice, end to end from the frame and from the GPU's own level l - 1 (which isolates the
decimation kernel); the gradients from the GPU's own intensity plane of the level.

Where a kernel filters a reflect-extended input it computed itself (the fused level-0 kernels smooth the mirrored frame
instead of mirroring the smoothed image), its values beyond the border are the same numbers in real arithmetic but not
in fp32: against the GPU's own plane, the outputs within the filter's radius of the image edge get an input error of
twice the level-0 bound; the interior reads the very values the kernel stored and is checked with none.

Every GPU case asserts which kernels ran (the context's launch profile), so that a case keeps testing the path it was
written for when a launcher changes its dispatch.  Run with -s to see each check's measured error / bound."""
import ctypes as C
import hashlib

import numpy as np
import pytest

U = 2.0 ** -24


# ---- float64 reference -----------------------------------------------------------------------------------------------------
def reflect_index(i, n):
    """SciPy's 'reflect' (half-sample symmetric: d c b a | a b c d | d c b a), repeated for any overshoot: period 2n."""
    i = np.mod(np.asarray(i), 2 * n)
    return np.where(i < n, i, 2 * n - 1 - i)


def conv1d(a, k, axis, start=0, step=1, count=None):
    """scipy.ndimage.convolve1d(a, k, axis, mode='reflect') in float64 for odd-length kernels (every KLT kernel is odd;
    SciPy moves the origin of even-length ones by one sample), evaluated at positions start + step * i only."""
    a = np.asarray(a, np.float64)
    k = np.asarray(k, np.float64)
    n, L = len(k), a.shape[axis]
    size1 = n // 2
    if count is None:
        count = len(range(start, L, step))
    pos = start + step * np.arange(count)
    fw = k[::-1]                         # convolution = correlation with the reversed taps: fw[j] multiplies a[x + j - size1]
    out = np.zeros(a.shape[:axis] + (count,) + a.shape[axis + 1:])
    for j in range(n):
        out += fw[j] * np.take(a, reflect_index(pos + j - size1, L), axis=axis)
    return out


def conv_separable(img, hk, vk):
    """_convolveSeparate: the horizontal kernel along rows first, then the vertical one along columns."""
    return conv1d(conv1d(img, hk, 1), vk, 0)


def gradients(img, g, d):
    """KLTComputeGradients: gradx = deriv_h o gauss_v, grady = gauss_h o deriv_v."""
    return conv_separable(img, d, g), conv_separable(img, g, d)


def pyramid_step(img, p, ss):
    """One level of KLTPyramid.Compute: smooth with p, keep pixel (ss * Y + ss / 2, ss * X + ss / 2); int(h / ss) x int(w / ss)."""
    h, w = img.shape
    t = conv1d(img, p, 1, ss // 2, ss, int(w / ss))
    return conv1d(t, p, 0, ss // 2, ss, int(h / ss))


def min_eigen_map(gx, gy, hw, bx, by, step):
    """float64 window sums of gx^2, gx gy, gy^2 and the minimum eigenvalue, laid out like the scan's output: candidate
    (x, y) for x in [bx, W - bx), y in [by, H - by), both with the given step.  Also returns max(gxx + gyy)."""
    gx, gy = np.asarray(gx, np.float64), np.asarray(gy, np.float64)
    H, W = gx.shape
    k = 2 * hw + 1

    def box(a):                          # box[i, j] = sum over rows i .. i + 2hw, columns j .. j + 2hw
        s = np.pad(a.cumsum(0).cumsum(1), ((1, 0), (1, 0)))
        return s[k:, k:] - s[:-k, k:] - s[k:, :-k] + s[:-k, :-k]
    gxx, gxy, gyy = box(gx * gx), box(gx * gy), box(gy * gy)
    lam = 0.5 * ((gxx + gyy) - np.sqrt((gxx - gyy) ** 2 + 4 * gxy ** 2))
    return lam[by - hw:H - by - hw:step, bx - hw:W - bx - hw:step], float((gxx + gyy).max())


def pass_bound(h, v, e_in, M):
    """Error bound of one fp32 separable pass (module docstring)."""
    A = float(np.abs(h).sum() * np.abs(v).sum())
    return A * e_in + (len(h) + len(v) + 4) * U * A * M


def taps_of(k):
    return np.array([k.taps[i] for i in range(k.n)], np.float64)


class Taps:
    """The four kernels of a klt_taps struct as float64 arrays."""

    def __init__(self, t):
        self.s, self.p = taps_of(t.smooth), taps_of(t.pyramid)
        self.g, self.d = taps_of(t.grad_gauss), taps_of(t.grad_deriv)
        self.key = tuple(np.concatenate([self.s, [np.nan], self.p, [np.nan], self.g, [np.nan], self.d]).tolist())


_REF_CACHE = {}


def reference_pyramid(frame, T, L, ss, smoothed=False):
    """float64 levels of one frame and the end-to-end bound of each (cached per frame, taps and geometry).  smoothed: the
    frame is level 0 itself (already-smoothed float input), exact."""
    key = (hashlib.sha1(np.ascontiguousarray(frame).tobytes()).hexdigest(), frame.shape, str(frame.dtype), T.key, L, ss, smoothed)
    hit = _REF_CACHE.get(key)
    if hit is None:
        f = np.asarray(frame, np.float64)
        if smoothed:
            levels, bounds = [f], [0.0]
        else:
            levels, bounds = [conv_separable(f, T.s, T.s)], [pass_bound(T.s, T.s, 0.0, float(np.abs(f).max()))]
        for _ in range(1, L):
            M = float(np.abs(levels[-1]).max()) + bounds[-1]
            levels.append(pyramid_step(levels[-1], T.p, ss))
            bounds.append(pass_bound(T.p, T.p, bounds[-1], M))
        if len(_REF_CACHE) > 256:
            _REF_CACHE.clear()
        hit = _REF_CACHE[key] = (levels, bounds)
    return hit


def edge_mask(in_shape, out_shape, r, ss=1):
    """Outputs (ss * Y + ss / 2, ss * X + ss / 2 of the input; ss = 1: the same pixel) whose radius-r window reaches past
    the input's border."""
    def axis(n, m):
        pos = ss * np.arange(m) + ss // 2
        return (pos - r < 0) | (pos + r >= n)
    return axis(in_shape[0], out_shape[0])[:, None] | axis(in_shape[1], out_shape[1])[None, :]


RATIOS = {}


def check(got, want, bound, label, kind):
    """max|got - want| <= bound; prints and records the ratio."""
    assert got.shape == want.shape, (label, got.shape, want.shape)
    assert np.isfinite(got).all(), label
    err = float(np.abs(got.astype(np.float64) - want).max()) if got.size else 0.0
    ratio = err / bound
    RATIOS[kind] = max(RATIOS.get(kind, 0.0), ratio)
    print("fp64 %-72s err %.3e  bound %.3e  err/bound %.3f" % (label, err, bound, ratio))
    assert err <= bound, "%s: max error %.4g above its bound %.4g (ratio %.3f)" % (label, err, bound, ratio)


@pytest.fixture(scope="module", autouse=True)
def _ratio_summary():
    yield
    if RATIOS:
        print("\nfp64 largest err/bound per stage: " + ", ".join("%s %.3f" % kv for kv in sorted(RATIOS.items())))


def check_split(got, want, bound, edge_bound, mask, label, kind):
    """check() with `bound` on the outputs off `mask` and `edge_bound` on those on it."""
    assert got.shape == want.shape, (label, got.shape, want.shape)
    check(got[~mask], want[~mask], bound, label + " interior", kind)
    if mask.any():
        check(got[mask], want[mask], edge_bound, label + " edge", kind)


def check_pyramid(pyr, image, frame, T, L, ss, label, fused0=False, fused01=False, grads=True, level0_exact=False):
    """Levels (end to end and from the GPU's own previous level) and, with grads, both gradient planes of every level of
    image `image` of a batch built from `frame`.  fused0: level-0 gradients came from stream_level0, which filters its own
    smoothed extension of the frame beyond the border; fused01: level 1 came from stream_level01, likewise.  level0_exact:
    level 0 is the input itself (already-smoothed float input)."""
    levels, bounds = reference_pyramid(frame, T, L, ss, smoothed=level0_exact)
    got = [pyr.download(0, lvl, image) for lvl in range(L)]
    if level0_exact:
        assert np.array_equal(got[0], frame), label
    for lvl in range(L):
        tag = "%s img%d L%d" % (label, image, lvl)
        if not (level0_exact and lvl == 0):
            check(got[lvl], levels[lvl], bounds[lvl], tag + " end-to-end", "level%d" % min(lvl, 1))
        if lvl >= 1:
            own = pyramid_step(got[lvl - 1], T.p, ss)
            M = float(np.abs(got[lvl - 1]).max())
            edge_e = 2 * bounds[0] if (lvl == 1 and fused01) else 0.0
            mask = edge_mask(got[lvl - 1].shape, got[lvl].shape, len(T.p) // 2, ss)
            check_split(got[lvl], own, pass_bound(T.p, T.p, 0.0, M), pass_bound(T.p, T.p, edge_e, M),
                        mask, tag + " from own L%d" % (lvl - 1), "decimation")
    if grads:
        r = max(len(T.g), len(T.d)) // 2
        for lvl in range(L):
            gx, gy = pyr.download(1, lvl, image), pyr.download(2, lvl, image)
            wx, wy = gradients(got[lvl], T.g, T.d)
            M = float(np.abs(got[lvl]).max())
            edge_e = 2 * bounds[0] if (lvl == 0 and fused0) else 0.0
            mask = edge_mask(got[lvl].shape, got[lvl].shape, r)
            for g, w, name in ((gx, wx, "gradx"), (gy, wy, "grady")):
                check_split(g, w, pass_bound(T.d, T.g, 0.0, M), pass_bound(T.d, T.g, edge_e, M), mask,
                            "%s img%d L%d %s" % (label, image, lvl, name), "gradients")
    return got


# ---- which kernels a build runs: the launchers' dispatch (klt_api.cu, klt_stream.cu), restated ------------------------------
def level_dims(W, H, L, ss):
    dims = [(W, H)]
    for _ in range(1, L):
        dims.append((int(dims[-1][0] / ss), int(dims[-1][1] / ss)))
    return dims


def grad_kernel(w, h):
    return "stream_grad" if w >= 16 and h >= 8 and w % 4 == 0 else "grad_pair"


def decimation_kernel(a, b, ss):
    (aw, ah), (bw, bh) = a, b
    if ss == 2 and bw >= 8 and bh >= 8 and aw >= 32 and ah >= 16 and aw % 4 == 0 and bw % 4 == 0:
        return "stream_down2"
    if ss == 4 and bw >= 8 and bh >= 8 and aw >= 64 and ah >= 32 and aw % 4 == 0 and bw % 4 == 0:
        return "stream_down4"
    return "pyr_down"


def expected_kernels(W, H, L, ss, n_smooth, windowed, align=8, source="u8"):
    """Kernel names a FAST (windowed=False) or FAST_WINDOWED build launches.  align: the largest of 8, 4, 1 that divides the
    frame pointer, the pitch and the frame stride.  source: 'u8', 'f32' or 'f32_smoothed'."""
    dims = level_dims(W, H, L, ss)
    ks, first, grads_from = set(), 1, 0
    streamable = n_smooth in (3, 5, 7, 9) and W >= 16 and H >= 16 and W % 4 == 0 and align % 4 == 0
    if source == "f32":
        ks.add("conv_sep_f32")
    elif source == "u8":
        if windowed:
            (bw, bh) = dims[1] if L >= 2 else (0, 0)
            if L >= 2 and ss == 2 and n_smooth == 5 and W >= 64 and H >= 32 and W % 8 == 0 and bw % 4 == 0 and bw >= 8 and \
                    bh >= 8 and align % 8 == 0:
                ks.add("stream_level01")
                first = 2
            else:
                ks.add("stream_smooth0" if streamable else "conv_sep_u8")
        elif streamable:
            ks.add("stream_level0")
            grads_from = 1
        else:
            ks.add("conv_sep_u8")
    for lvl in range(first, L):
        ks.add(decimation_kernel(dims[lvl - 1], dims[lvl], ss))
    if not windowed:
        for lvl in range(grads_from, L):
            ks.add(grad_kernel(*dims[lvl]))
    return ks


def profiled(ctx, fn):
    """Runs fn with the context's launch profile on; returns {kernel name: dict(launches=...)}."""
    ctx.profile(True)
    ctx.profile_reset()
    try:
        fn()
        return ctx.profile_read()
    finally:
        ctx.profile(False)


def make_tc(**kw):
    from pyfeaturetrack_b200 import klt
    tc = klt.KLT_TrackingContext()
    for k, v in kw.items():
        setattr(tc, k, v)
    tc.KLTUpdateTCBorder()
    return tc


def taps_for(**kw):
    from pyfeaturetrack_b200 import trackFeatures
    t = trackFeatures._taps_for_one_image(make_tc(**kw))
    return t, Taps(t)


def random_frames(seed, B, H, W):
    return np.random.default_rng(seed).integers(0, 256, (B, H, W), dtype=np.uint8)


# ---- CPU: the reference against the oracle (which matches the original project bit for bit) ----------------------------------
# The oracle rounds to float32 once per 1-D pass and accumulates in double, so one separable pass of it differs from the
# float64 reference by at most u |h-pass| + (sum|v| u |h-pass| + u |out|) <= 2 u A M; 3 u A M leaves room for its double sums.
def oracle_bound(h, v, e_in, M):
    A = float(np.abs(h).sum() * np.abs(v).sum())
    return A * e_in + 3 * U * A * M


def test_reference_conv_matches_oracle_orientation_and_pass_order(oracle):
    """Non-symmetric taps of different lengths: a flipped kernel or swapped passes would miss by far more than rounding."""
    rng = np.random.default_rng(3)
    img = (rng.random((20, 31)) * 100).astype(np.float32)
    hk, vk = rng.random(7) - 0.3, rng.random(5) - 0.3
    want = oracle.conv_separable(img, hk, vk)
    got = conv_separable(img, hk, vk)
    b = oracle_bound(hk, vk, 0.0, float(np.abs(img).max()))
    assert np.abs(got - want).max() <= b
    assert np.abs(conv_separable(img, hk[::-1], vk) - want).max() > 1e3 * b
    assert np.abs(conv_separable(img, vk, hk) - want).max() > 1e3 * b


@pytest.mark.parametrize("shape", [(20, 31), (3, 40), (1, 9)])
def test_reference_conv_matches_oracle_kernel_wider_than_image(oracle, shape):
    """43 / 51 taps on images of 20, 3 and 1 rows: the border is reflected again and again (and a 1-pixel line is constant)."""
    rng = np.random.default_rng(shape[0])
    img = (rng.random(shape) * 255).astype(np.float32)
    g, d = oracle.compute_kernels(7.2)
    for hk, vk in ((d, g), (g, d), (g, g)):
        b = oracle_bound(hk, vk, 0.0, float(np.abs(img).max()))
        assert np.abs(conv_separable(img, hk, vk) - oracle.conv_separable(img, hk, vk)).max() <= b


def test_reference_gradients_match_oracle(oracle):
    rng = np.random.default_rng(5)
    img = (rng.random((77, 123)) * 255).astype(np.float32)
    cache = oracle.KernelCache()
    cache.compute(1.0)
    g, d = oracle.compute_kernels(1.0)
    want_x, want_y = oracle.gradients(img, 1.0, cache)
    got_x, got_y = gradients(img, g, d)
    b = oracle_bound(d, g, 0.0, float(np.abs(img).max()))
    assert np.abs(got_x - want_x).max() <= b and np.abs(got_y - want_y).max() <= b


@pytest.mark.parametrize("ss,L,shape,win", [(2, 3, (101, 157), 7), (4, 3, (203, 301), 11), (8, 2, (211, 333), 5)])
def test_reference_pyramid_matches_oracle(oracle, ss, L, shape, win):
    """oracle.image_pyramids against the reference fed with the klt_taps struct the GPU gets: the taps agree, and the levels
    and gradients differ by the oracle's per-pass rounding only."""
    kw = dict(nPyramidLevels=L, subsampling=ss, window_width=win, window_height=win)
    p = oracle.Params(**kw)
    _, T = taps_for(**kw)
    frame = random_frames(ss * 100 + L, 1, *shape)[0]
    want_lv, want_gx, want_gy = oracle.image_pyramids(p, frame)
    levels, _ = reference_pyramid(frame, T, L, ss)
    e = oracle_bound(T.s, T.s, 0.0, 255.0)
    for lvl in range(L):
        if lvl:
            e = oracle_bound(T.p, T.p, e, float(np.abs(levels[lvl - 1]).max()) + e)
        assert want_lv[lvl].shape == levels[lvl].shape
        assert np.abs(levels[lvl] - want_lv[lvl]).max() <= e, lvl
        wx, wy = gradients(want_lv[lvl], T.g, T.d)
        b = oracle_bound(T.d, T.g, 0.0, float(np.abs(want_lv[lvl]).max()))
        assert np.abs(wx - want_gx[lvl]).max() <= b and np.abs(wy - want_gy[lvl]).max() <= b, lvl


def test_pass_bound_catches_a_tap_scale_of_four_ppm():
    """The GPU cases below are meant to catch taps off by a few parts per million: on a random u8 frame such a kernel
    misses the level-0 bound by a wide margin, where the 1e-5 * 255 image tolerance of the older tests does not notice."""
    _, T = taps_for(nPyramidLevels=2, subsampling=2)
    frame = random_frames(9, 1, 64, 96)[0].astype(np.float64)
    exact = conv_separable(frame, T.s, T.s)
    off = conv_separable(frame, T.s * (1 + 4e-6), T.s)
    b = pass_bound(T.s, T.s, 0.0, 255.0)
    assert np.abs(off - exact).max() > 1.5 * b
    assert np.abs(off - exact).max() < 1e-5 * 255.0


# ---- GPU cases --------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _quiet():
    from pyfeaturetrack_b200 import selectGoodFeatures, trackFeatures
    selectGoodFeatures.KLT_verbose = 0
    trackFeatures.KLT_verbose = 0
    yield


def build_and_check(ctx, frames, win, L, ss, windowed, label, pitch=None, frame_stride=None, src=None, align=8, grads=True):
    """Builds `frames` (or `src` laid out with pitch / frame_stride) into one pyramid batch, asserts the kernels and checks
    every image."""
    from pyfeaturetrack_b200 import _capi
    B, H, W = frames.shape
    t, T = taps_for(nPyramidLevels=L, subsampling=ss, window_width=win, window_height=win)
    prec = _capi.PRECISION_FAST_WINDOWED if windowed else _capi.PRECISION_FAST
    pyr = _capi.Pyramid(ctx, W, H, L, ss, B)
    try:
        ran = profiled(ctx, lambda: pyr.build_u8(frames if src is None else src, t, prec, pitch, frame_stride))
        want = expected_kernels(W, H, L, ss, len(T.s), windowed, align)
        assert set(ran) == want, (label, sorted(ran), sorted(want))
        for b in range(B):
            check_pyramid(pyr, b, frames[b], T, L, ss, label, fused0="stream_level0" in ran, fused01="stream_level01" in ran,
                          grads=grads)
    finally:
        pyr.close()
    return ran


@gpu
@pytest.mark.parametrize("win,ss,L,H,W,B", [
    (5, 2, 3, 97, 132, 3),       # smoother radius 1
    (7, 2, 3, 270, 488, 3),      # radius 2; level 2 is 122 wide: pyr_down and grad_pair
    (11, 2, 3, 200, 480, 2),     # radius 3; stream_down2 twice
    (11, 2, 2, 135, 244, 3),
    (15, 2, 3, 200, 360, 2),     # radius 4
    (13, 4, 3, 270, 480, 2),     # stream_down4, then pyr_down
    (9, 8, 2, 360, 488, 2),      # subsampling 8: pyr_down
    (3, 2, 2, 120, 160, 2),      # 1-tap smoother: conv_sep_u8
    (17, 2, 2, 97, 132, 2),      # 11-tap smoother: conv_sep_u8
])
def test_fast_u8_build(gpu_ctx, win, ss, L, H, W, B):
    """KLT_PRECISION_FAST from u8 frames: stream_level0<RS> for RS = 1..4 (or the conv_sep_u8 fallback), the decimation of
    each subsampling, and stream_grad or grad_pair per level."""
    frames = random_frames(win * 1000 + H, B, H, W)
    build_and_check(gpu_ctx, frames, win, L, ss, False, "fast w%d ss%d %dx%d" % (win, ss, H, W))


LEVEL01_SHAPES = [(32, 64), (33, 72), (47, 120), (97, 240), (135, 248), (270, 320), (33, 488), (47, 640), (97, 720),
                  (135, 960), (270, 1000), (32, 1280), (1080, 1920), (1080, 1928)]


@gpu
@pytest.mark.parametrize("H,W", LEVEL01_SHAPES)
def test_windowed_level01_build(gpu_ctx, H, W):
    """KLT_PRECISION_FAST_WINDOWED through stream_level01 at the widths its column bookkeeping is modelled for (one strip, a
    strip pair whose second strip lies outside the image, widths that are not multiples of 240) and heights from its 32-row
    minimum up; levels >= 2 by the decimation, and the gradient planes built on demand."""
    L = 3 if H >= 64 else 2
    frames = random_frames(H * 7 + W, 2, H, W)
    build_and_check(gpu_ctx, frames, 7, L, 2, True, "level01 %dx%d" % (H, W))


@gpu
@pytest.mark.parametrize("W,H,win,L", [(16, 16, 5, 1), (120, 33, 11, 1), (124, 47, 15, 2), (132, 97, 5, 2), (240, 97, 11, 2),
                                       (244, 135, 11, 2), (964, 270, 15, 1), (964, 47, 7, 1), (1924, 1080, 5, 2)])
def test_windowed_smooth0_build(gpu_ctx, W, H, win, L):
    """KLT_PRECISION_FAST_WINDOWED through stream_smooth0x2<RS> (RS = 1..4): one strip, an odd number of strips, widths the
    fused level-0/1 kernel declines; then the decimation and the gradient planes built on demand."""
    frames = random_frames(W * 3 + H + win, 2, H, W)
    build_and_check(gpu_ctx, frames, win, L, 2, True, "smooth0 w%d %dx%d" % (win, H, W))


@gpu
@pytest.mark.parametrize("windowed", [False, True])
@pytest.mark.parametrize("H,W,batches", [(97, 248, (64, 3, 1)), (1080, 1920, (8, 1))])
def test_segment_height_follows_the_batch(gpu_ctx, windowed, H, W, batches):
    """The launchers pick the segment height from the SM count and the batch size: the same frames built as batches of
    different sizes are cut into different segments, and every image of every batch must meet its bound."""
    frames = random_frames(H + W, batches[0], H, W)
    for B in batches:
        build_and_check(gpu_ctx, np.ascontiguousarray(frames[:B]), 7, 3, 2, windowed,
                        "%s batch %d %dx%d" % ("windowed" if windowed else "fast", B, H, W))


def _strided(frames, pitch, stride, offset=0):
    B, H, W = frames.shape
    buf = np.zeros(offset + (B - 1) * stride + (H - 1) * pitch + W, np.uint8)
    for b in range(B):
        for y in range(H):
            buf[offset + b * stride + y * pitch:offset + b * stride + y * pitch + W] = frames[b, y]
    return buf


@gpu
@pytest.mark.parametrize("windowed", [False, True])
@pytest.mark.parametrize("layout", ["contiguous", "pitch+4", "stride+4", "pitch+1", "device+4", "device+1"])
def test_frame_layout_fallbacks(gpu_ctx, windowed, layout):
    """Identical frames in layouts the streaming kernels accept or decline: the fused level-0/1 kernel needs 8-byte
    alignment of pointer, pitch and frame stride, the other streaming kernels 4 bytes, and with neither conv_sep_u8 runs.
    Whatever ran, the images meet the same bounds."""
    B, H, W = 2, 200, 360
    frames = random_frames(77, B, H, W)
    pitch, stride, off = W, H * W, 0
    if layout == "pitch+4":
        pitch += 4
    elif layout == "pitch+1":
        pitch += 1
    elif layout == "stride+4":
        stride += 4
    elif layout.startswith("device"):
        off = int(layout[-1])
    if layout.startswith("pitch"):
        stride = H * pitch
    align = 8
    for v in (pitch, stride, off):
        while v % align:
            align //= 2
    buf = _strided(frames, pitch, stride)
    label = "%s %s" % ("windowed" if windowed else "fast", layout)
    if off:
        d = gpu_ctx.device_alloc(buf.size + 64)
        try:
            gpu_ctx.memcpy(d + off, buf, buf.size)
            build_and_check(gpu_ctx, frames, 7, 3, 2, windowed, label, pitch, stride, src=d + off, align=align)
        finally:
            gpu_ctx.sync()
            gpu_ctx.device_free(d)
    else:
        build_and_check(gpu_ctx, frames, 7, 3, 2, windowed, label, pitch, stride, src=buf, align=align)


@gpu
@pytest.mark.parametrize("already_smoothed", [0, 1])
@pytest.mark.parametrize("H,W", [(120, 160), (97, 134)])
def test_f32_input_build(gpu_ctx, already_smoothed, H, W):
    """klt_pyr_build_f32 in FAST mode with values in [-1000, 1000] (off the u8 grid) in a buffer whose pitch exceeds the
    width; the bound scales with max|input|.  Already-smoothed input becomes level 0 unchanged."""
    from pyfeaturetrack_b200 import _capi
    B, L, ss, pitch = 2, 3, 2, W + 5
    imgs = np.random.default_rng(H + already_smoothed).uniform(-1000, 1000, (B, H, W)).astype(np.float32)
    buf = np.zeros((B, H, pitch), np.float32)
    buf[:, :, :W] = imgs
    t, T = taps_for(nPyramidLevels=L, subsampling=ss)
    pyr = _capi.Pyramid(gpu_ctx, W, H, L, ss, B)
    try:
        ran = profiled(gpu_ctx, lambda: pyr.build_f32(buf, t, _capi.PRECISION_FAST, already_smoothed, pitch, H * pitch))
        want = expected_kernels(W, H, L, ss, len(T.s), False, source="f32_smoothed" if already_smoothed else "f32")
        assert set(ran) == want, (sorted(ran), sorted(want))
        for b in range(B):
            check_pyramid(pyr, b, imgs[b], T, L, ss, "f32 smoothed=%d %dx%d" % (already_smoothed, H, W),
                          level0_exact=bool(already_smoothed))
    finally:
        pyr.close()


@gpu
@pytest.mark.parametrize("windowed", [False, True])
@pytest.mark.parametrize("B", [5, 17])
def test_chunked_host_pairs(gpu_ctx, oracle, windowed, B):
    """klt_track_pairs_u8 with host frames builds the batch in chunks (5 -> 3 + 2, 17 -> 5 + 5 + 5 + 2), each chunk's
    kernels writing images first .. first + count - 1.  Every image of both pyramids meets its bound, and the feature lists
    are bit-equal to the same pairs built one at a time and tracked with klt_track_features."""
    from pyfeaturetrack_b200 import _capi, synth, selectGoodFeatures as sgf
    lib = _capi.lib()
    H, W, L, ss, n = 120, 160, 2, 2, 32
    kw = dict(nPyramidLevels=L, subsampling=ss, max_residue=10.0)
    tc = make_tc(**kw)
    p = oracle.Params(**kw)
    t, T = taps_for(**kw)
    params = sgf.make_params(tc)
    prec = _capi.PRECISION_FAST_WINDOWED if windowed else _capi.PRECISION_FAST
    f1, f2 = np.empty((B, H, W), np.uint8), np.empty((B, H, W), np.uint8)
    xs, ys, vs = np.empty((B, n)), np.empty((B, n)), np.empty((B, n), np.int32)
    for b in range(B):
        f1[b], f2[b] = synth.frame_pair(H, W, seed=300 + b, shift=(0.8, -1.1))
        xs[b], ys[b], vs[b] = oracle.select_good_features(p, f1[b], n)
    start = (xs.copy(), ys.copy(), vs.copy())
    p1, p2 = _capi.Pyramid(gpu_ctx, W, H, L, ss, B), _capi.Pyramid(gpu_ctx, W, H, L, ss, B)
    try:
        ran = profiled(gpu_ctx, lambda: gpu_ctx.check(lib.klt_track_pairs_u8(
            gpu_ctx.handle, C.byref(params), C.byref(t), prec, p1.handle, p2.handle, f1.ctypes.data, f2.ctypes.data, W, W * H,
            n, xs.ctypes.data, ys.ctypes.data, vs.ctypes.data)))
        nchunks = 2 if B < 16 else 4
        first_kernel = "stream_level01" if windowed else "stream_level0"
        assert ran[first_kernel]["launches"] == 2 * nchunks, (first_kernel, ran[first_kernel])
        assert "conv_sep_u8" not in ran
        for pyr, frames, name in ((p1, f1, "frames1"), (p2, f2, "frames2")):
            for b in range(B):
                check_pyramid(pyr, b, frames[b], T, L, ss, "pairs B=%d %s %s" % (B, "windowed" if windowed else "fast", name),
                              fused0=not windowed, fused01=windowed)
    finally:
        p1.close(); p2.close()
    for b in range(B):
        q1, q2 = _capi.Pyramid(gpu_ctx, W, H, L, ss, 1), _capi.Pyramid(gpu_ctx, W, H, L, ss, 1)
        try:
            q1.build_u8(f1[b], t, prec)
            q2.build_u8(f2[b], t, prec)
            x, y, v = start[0][b].copy(), start[1][b].copy(), start[2][b].copy()
            gpu_ctx.check(lib.klt_track_features(gpu_ctx.handle, C.byref(params), q1.handle, q2.handle, n, x.ctypes.data,
                                                 y.ctypes.data, v.ctypes.data, None))
        finally:
            q1.close(); q2.close()
        assert np.array_equal(vs[b], v) and np.array_equal(xs[b], x) and np.array_equal(ys[b], y), b
    assert (vs == 0).mean() > 0.25           # the pairs do get tracked


def eigen_case(ctx, frames, win, skip, label, border=None):
    """klt_eigen_map_batch (SELECT_FAST) on a FAST_WINDOWED pyramid of `frames`, per image against the float64 map of the
    GPU's own level-0 image; asserts which of the two fused kernels ran and that no gradient plane or table was built."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf
    B, H, W = frames.shape
    tc = make_tc(window_width=win, window_height=win, nPyramidLevels=1, subsampling=2, nSkippedPixels=skip)
    if border is not None:
        tc.borderx = tc.bordery = border
    t, T = taps_for(window_width=win, window_height=win, nPyramidLevels=1, subsampling=2)
    params = sgf.make_params(tc)
    pyr = _capi.Pyramid(ctx, W, H, 1, 2, B)
    try:
        pyr.build_u8(frames, t, _capi.PRECISION_FAST_WINDOWED)
        nx, ny = C.c_int(), C.c_int()
        ctx.check(_capi.lib().klt_eigen_map_batch(ctx.handle, C.byref(params), pyr.handle, _capi.SELECT_FAST, None,
                                                  C.byref(nx), C.byref(ny)))
        assert nx.value > 0 and ny.value > 0
        got = np.empty((B, ny.value, nx.value), np.float32)
        ran = profiled(ctx, lambda: ctx.check(_capi.lib().klt_eigen_map_batch(
            ctx.handle, C.byref(params), pyr.handle, _capi.SELECT_FAST, got.ctypes.data, C.byref(nx), C.byref(ny))))
        hw = int(win / 2)
        # the quad kernel ("eigen_fast") serves half-windows up to 3 on images of 16 rows or more, the plain one
        # ("eigen_fast_rows") everything else
        assert set(ran) == {"eigen_fast" if hw <= 3 and H >= 16 else "eigen_fast_rows"}, sorted(ran)
        bx, by = int(max(tc.borderx, win / 2)), int(max(tc.bordery, win / 2))
        for b in range(B):
            gx, gy = gradients(pyr.download(0, 0, b), T.g, T.d)
            want, scale = min_eigen_map(gx, gy, hw, bx, by, skip + 1)
            check(got[b], want, 2e-5 * scale, "%s img%d" % (label, b), "eigen")
    finally:
        pyr.close()


@gpu
@pytest.mark.parametrize("win,skip,B,H,W", [(3, 0, 1, 130, 203), (5, 1, 3, 130, 203), (7, 3, 3, 97, 250), (7, 0, 3, 120, 160),
                                            (9, 0, 3, 97, 250), (11, 1, 1, 120, 161), (13, 3, 3, 120, 161), (15, 0, 1, 150, 246),
                                            (15, 1, 3, 90, 128)])
def test_fused_eigen_map(gpu_ctx, win, skip, B, H, W):
    """The fused eigenvalue pass for half-windows 1..7 (the quad kernels up to 3, the plain ones above), skipped pixels,
    batches and widths that are not multiples of 4.  Bound: the 2e-5 * max(gxx + gyy) of the existing map test."""
    eigen_case(gpu_ctx, random_frames(win * 10 + skip + H, B, H, W), win, skip, "eigen w%d skip%d B%d %dx%d" % (win, skip, B, H, W))


@gpu
@pytest.mark.parametrize("win", [3, 5, 7])
def test_fused_eigen_map_short_image(gpu_ctx, win):
    """Images under 16 rows take the plain kernel even for windows up to 7x7 (the quad kernel reflects rows only once);
    with the border set to the smallest the selection accepts, such an image still has candidate rows."""
    eigen_case(gpu_ctx, random_frames(win, 2, 14, 61), win, 0, "eigen short w%d" % win, border=int(win / 2) + 1)
