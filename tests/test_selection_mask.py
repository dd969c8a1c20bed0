"""Selection masks (beyond the reference; cf. the mask of OpenCV's goodFeaturesToTrack): klt_select_good_features_batch_masked,
klt_sequence_set_mask and tc.selection_mask.

A masked-out candidate is never selected and suppresses nothing.  The walk ignores values below min_eigenvalue (clamped to
at least 1) and sorts on (val, x, y), so that is the reference's selection with the candidate's eigenvalue set to 0.  The
reference is composed on the oracle that way: scan (or the GPU's own FAST map), zero the masked candidates, walk with
orc_select_from_scan.  STRICT pyramids with STRICT selection must reproduce it bit for bit (==)."""
import ctypes as C

import numpy as np
import pytest

gpu = pytest.mark.gpu


# ---- reference composition -------------------------------------------------------------------------------------------------
def geometry(p):
    """(bx, by, hw, hh, step) exactly as selectGoodFeatures.py:168-169,215-230 (true division, then truncation)."""
    hw, hh = p.window_width / 2, p.window_height / 2
    return int(max(p.borderx, hw)), int(max(p.bordery, hh)), int(hw), int(hh), p.nSkippedPixels + 1


def masked_walk(oracle, p, val, W, H, n, mask, existing=None):
    """Sort + _enforceMinimumDistance on the eigenvalue map `val` [ny, nx] with every candidate on a mask == 0 pixel set to 0."""
    bx, by, _, _, step = geometry(p)
    ny, nx = val.shape
    xs, ys = bx + step * np.arange(nx), by + step * np.arange(ny)
    v = np.array(val, np.float32)
    if mask is not None:
        v[np.asarray(mask)[np.ix_(ys, xs)] == 0] = 0.0
    if existing is None:
        fx, fy, fv, overwrite = np.full(n, -1.0), np.full(n, -1.0), np.full(n, -1, np.int32), 1
    else:
        fx, fy, fv = (np.array(existing[0], np.float64), np.array(existing[1], np.float64), np.array(existing[2], np.int32))
        overwrite = 0
    used = oracle.lib().orc_select_from_scan(oracle._f(v), nx, ny, bx, by, p.nSkippedPixels, W, H, max(p.mindist, 0),
                                             float(p.min_eigenvalue), overwrite, n, oracle._d(fx), oracle._d(fy), oracle._i(fv))
    assert used >= 0
    return fx, fy, fv


def masked_select(oracle, p, gx, gy, n, mask, existing=None):
    """_KLTSelectGoodFeatures from the scan onwards on level-0 gradients, restricted to `mask`."""
    bx, by, hw, hh, _ = geometry(p)
    val, _, _ = oracle.scan_good_features(gx, gy, bx, by, hw, hh, p.nSkippedPixels)
    H, W = gx.shape
    return masked_walk(oracle, p, val, W, H, n, mask, existing)


def make_mask(H, W, seed, border=20):
    """Cells of 16 px of which about a third are masked out, a burned-in 'timestamp' block, a black border; allowed pixels
    carry arbitrary nonzero values."""
    rng = np.random.default_rng(seed)
    cells = rng.random(((H + 15) // 16, (W + 15) // 16)) >= 0.35
    m = np.kron(cells, np.ones((16, 16), bool))[:H, :W].copy()
    m[H // 8:H // 8 + 24, W // 2:W // 2 + 120] = False
    m[:border] = m[-border:] = False
    m[:, :border] = m[:, -border:] = False
    vals = rng.integers(1, 256, size=(H, W)).astype(np.uint8)
    return np.where(m, vals, 0).astype(np.uint8)


def knock_out(x, y, v, every=3):
    x, y, v = np.array(x, np.float64), np.array(y, np.float64), np.array(v, np.int32)
    x[..., ::every] = -1.0; y[..., ::every] = -1.0; v[..., ::every] = -1
    return x, y, v


def frames_for(H, W, B, seed):
    from pyfeaturetrack_b200 import synth
    return [synth.frames(H, W, [(0.0, 0.0)], seed=seed + s)[0] for s in range(B)]


def eq(got, want):
    for a, b in zip(got, want):
        assert np.array_equal(np.asarray(a), np.asarray(b))


# ---- CPU: the composition itself -------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def scene(oracle):
    from pyfeaturetrack_b200 import synth
    p = oracle.Params(nPyramidLevels=2, subsampling=2)
    f = synth.frames(240, 320, [(0.0, 0.0)], seed=7)[0]
    _, gxs, gys = oracle.image_pyramids(p, f)
    return p, gxs[0], gys[0]


def test_all_ones_mask_leaves_the_oracle_selection_unchanged(oracle, scene):
    p, gx, gy = scene
    want = oracle.select_from_gradients(p, gx, gy, 150)[:3]
    eq(masked_select(oracle, p, gx, gy, 150, np.ones(gx.shape, np.uint8)), want)
    kx, ky, kv = knock_out(*want)
    eq(masked_select(oracle, p, gx, gy, 150, np.full(gx.shape, 9, np.uint8), existing=(kx, ky, kv)),
       oracle.select_from_gradients(p, gx, gy, 150, existing=(kx, ky, kv))[:3])


def test_masked_composition_places_features_on_allowed_pixels_only(oracle, scene):
    p, gx, gy = scene
    H, W = gx.shape
    mask = make_mask(H, W, 1)
    x, y, v = masked_select(oracle, p, gx, gy, 150, mask)
    ok = v >= 0
    assert ok.sum() > 50
    assert (mask[y[ok].astype(int), x[ok].astype(int)] != 0).all()
    # replacement: survivors stay where they are (also on masked pixels); only new features obey the mask
    full = oracle.select_from_gradients(p, gx, gy, 150)[:3]
    kx, ky, kv = knock_out(*full)
    rx, ry, rv = masked_select(oracle, p, gx, gy, 150, mask, existing=(kx, ky, kv))
    kept = kv >= 0
    eq((rx[kept], ry[kept], rv[kept]), (kx[kept], ky[kept], kv[kept]))
    assert (mask[ky[kept].astype(int), kx[kept].astype(int)] == 0).any()
    new = ~kept & (rv >= 0)
    assert new.any() and (mask[ry[new].astype(int), rx[new].astype(int)] != 0).all()


def test_mask_over_the_best_candidates_changes_the_result(oracle, scene):
    p, gx, gy = scene
    x, y, v = oracle.select_from_gradients(p, gx, gy, 150)[:3]
    mask = np.ones(gx.shape, np.uint8)
    for f in range(10):                       # the ten best features' pixels
        mask[int(y[f]), int(x[f])] = 0
    mx, my, mv = masked_select(oracle, p, gx, gy, 150, mask)
    assert not (np.array_equal(mx, x) and np.array_equal(my, y) and np.array_equal(mv, v))
    assert not {(int(a), int(b)) for a, b in zip(x[:10], y[:10])} & {(int(a), int(b)) for a, b in zip(mx, my)}


def test_selection_mask_default_and_bindings():
    from pyfeaturetrack_b200 import klt, _capi
    assert klt.KLT_TrackingContext().selection_mask is None
    for name in ("klt_select_good_features_batch_masked", "klt_sequence_set_mask"):
        assert name in _capi.SIGNATURES


# ---- GPU -------------------------------------------------------------------------------------------------------------------
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


def lay_out(masks, pitch, shared, gap=48, seed=0):
    """masks [(H, W)] -> (flat uint8 buffer, pitch, stride): row padding and the gaps between images hold 0 / 255 garbage."""
    rng = np.random.default_rng(seed)
    H, W = masks[0].shape
    stride = 0 if shared else H * pitch + gap
    n_img = 1 if shared else len(masks)
    buf = (rng.integers(0, 2, size=max(stride, H * pitch) * n_img) * 255).astype(np.uint8)
    for b in range(n_img):
        img = buf[b * stride:b * stride + H * pitch].reshape(H, pitch)
        img[:, :W] = masks[b]
    return buf, pitch, stride


def select_masked(ctx, tc, pyr, n, replace, mode, layout, existing=None, device=False):
    """klt_select_good_features_batch_masked (layout None: mask NULL) with host feature arrays [batch][n]."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf
    B = pyr.batch
    if existing is None:
        x, y, v = np.full((B, n), -1.0), np.full((B, n), -1.0), np.full((B, n), -1, np.int32)
    else:
        x, y, v = (np.array(existing[0], np.float64), np.array(existing[1], np.float64), np.array(existing[2], np.int32))
    params = sgf.make_params(tc)
    d = None
    if layout is None:
        mp, pitch, stride = None, 0, 0
    else:
        buf, pitch, stride = layout
        mp = buf.ctypes.data
        if device:
            d = ctx.device_alloc(buf.nbytes)
            ctx.memcpy(d, buf, buf.nbytes)
            mp = d
    ctx.check(_capi.lib().klt_select_good_features_batch_masked(ctx.handle, C.byref(params), pyr.handle, n, 1 if replace else 0,
                                                               mode, mp, pitch, stride, x.ctypes.data, y.ctypes.data,
                                                               v.ctypes.data))
    if d is not None:
        ctx.sync()
        ctx.device_free(d)
    return x, y, v


@gpu
@pytest.mark.parametrize("shape,B,n", [((240, 320), 3, 150), ((1080, 1920), 2, 1000)])
def test_batch_masked_strict_equals_composition(gpu_ctx, oracle, _quiet, shape, B, n):
    """Per-image masks and one shared mask (stride 0), pitch == w (16-byte path) and pitch > w (byte path), host and device
    masks, SELECTING_ALL and REPLACING_SOME: every image == the masked composition, slots included."""
    from pyfeaturetrack_b200 import _capi
    H, W = shape
    kw = dict(nPyramidLevels=3, subsampling=2)
    tc, p = make_tc(**kw), oracle.Params(**kw)
    frames = frames_for(H, W, B, 60)
    pyr = build_batch(gpu_ctx, tc, frames, _capi.PRECISION_STRICT)
    grads = [oracle.image_pyramids(p, f) for f in frames]
    grads = [(g[1][0], g[2][0]) for g in grads]
    masks = [make_mask(H, W, 10 + b) for b in range(B)]
    unmasked = [oracle.select_from_gradients(p, gx, gy, n)[:3] for gx, gy in grads]
    existing = knock_out(np.stack([u[0] for u in unmasked]), np.stack([u[1] for u in unmasked]),
                         np.stack([u[2] for u in unmasked]))
    cases = [(False, W, False), (False, W + 37, True), (True, W, True), (True, W + 37, False)]
    if H > 500:
        cases = [(False, W, False), (True, W + 37, True)]
    for shared, pitch, device in cases:
        use = [masks[0]] * B if shared else masks
        layout = lay_out(use[:1] if shared else use, pitch, shared, seed=pitch)
        for replace in (False, True):
            ex = existing if replace else None
            got = select_masked(gpu_ctx, tc, pyr, n, replace, _capi.SELECT_STRICT, layout, existing=ex, device=device)
            for b, (gx, gy) in enumerate(grads):
                want = masked_select(oracle, p, gx, gy, n, use[b], existing=None if ex is None else (ex[0][b], ex[1][b], ex[2][b]))
                eq((got[0][b], got[1][b], got[2][b]), want)
                if not replace:
                    assert not np.array_equal(want[0], unmasked[b][0])
    pyr.close()


@gpu
def test_fast_masked_selection_equals_masked_walk_of_the_gpu_map(gpu_ctx, oracle, _quiet):
    """FAST selection (fused pass): the GPU's own FAST map, masked and walked by the oracle, == the masked FAST selection."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf
    H, W, B, n = 480, 640, 2, 300
    kw = dict(nPyramidLevels=3, subsampling=2)
    tc, p = make_tc(**kw), oracle.Params(**kw)
    frames = frames_for(H, W, B, 80)
    pyr = build_batch(gpu_ctx, tc, frames, _capi.PRECISION_FAST_WINDOWED)
    params = sgf.make_params(tc)
    nx, ny = C.c_int(), C.c_int()
    gpu_ctx.check(_capi.lib().klt_eigen_map_batch(gpu_ctx.handle, C.byref(params), pyr.handle, _capi.SELECT_FAST, None,
                                                  C.byref(nx), C.byref(ny)))
    vmap = np.empty((B, ny.value, nx.value), np.float32)
    gpu_ctx.check(_capi.lib().klt_eigen_map_batch(gpu_ctx.handle, C.byref(params), pyr.handle, _capi.SELECT_FAST,
                                                  vmap.ctypes.data, C.byref(nx), C.byref(ny)))
    masks = [make_mask(H, W, 30 + b) for b in range(B)]
    layout = lay_out(masks, W, False)
    got = select_masked(gpu_ctx, tc, pyr, n, False, _capi.SELECT_FAST, layout)
    want = [masked_walk(oracle, p, vmap[b], W, H, n, masks[b]) for b in range(B)]
    for b in range(B):
        eq((got[0][b], got[1][b], got[2][b]), want[b])
    ex = knock_out(*got)
    got = select_masked(gpu_ctx, tc, pyr, n, True, _capi.SELECT_FAST, layout, existing=ex)
    for b in range(B):
        eq((got[0][b], got[1][b], got[2][b]), masked_walk(oracle, p, vmap[b], W, H, n, masks[b],
                                                          existing=(ex[0][b], ex[1][b], ex[2][b])))
    pyr.close()


@gpu
@pytest.mark.parametrize("mode", ["strict", "fast"])
def test_edge_masks(gpu_ctx, oracle, _quiet, mode):
    """All ones == the unmasked call bit for bit in both selection modes; all zeros leaves every slot KLT_NOT_FOUND
    (SELECTING_ALL) and every lost slot lost (REPLACING_SOME)."""
    from pyfeaturetrack_b200 import _capi
    H, W, B, n = 240, 320, 2, 150
    kw = dict(nPyramidLevels=2, subsampling=2)
    tc = make_tc(**kw)
    sel = _capi.SELECT_STRICT if mode == "strict" else _capi.SELECT_FAST
    prec = _capi.PRECISION_STRICT if mode == "strict" else _capi.PRECISION_FAST_WINDOWED
    pyr = build_batch(gpu_ctx, tc, frames_for(H, W, B, 90), prec)
    ones, zeros = lay_out([np.ones((H, W), np.uint8)], W, True), lay_out([np.zeros((H, W), np.uint8)], W + 5, True)
    plain = select_masked(gpu_ctx, tc, pyr, n, False, sel, None)
    eq(select_masked(gpu_ctx, tc, pyr, n, False, sel, ones), plain)
    ex = knock_out(*plain)
    plain_r = select_masked(gpu_ctx, tc, pyr, n, True, sel, None, existing=ex)
    eq(select_masked(gpu_ctx, tc, pyr, n, True, sel, ones, existing=ex), plain_r)
    x, y, v = select_masked(gpu_ctx, tc, pyr, n, False, sel, zeros)
    assert (v == -1).all() and (x == -1.0).all() and (y == -1.0).all()
    eq(select_masked(gpu_ctx, tc, pyr, n, True, sel, zeros, existing=ex), ex)
    # a pitch smaller than the width is refused
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf
    params = sgf.make_params(tc)
    xx, yy, vv = np.full((B, n), -1.0), np.full((B, n), -1.0), np.full((B, n), -1, np.int32)
    buf = ones[0]
    assert _capi.lib().klt_select_good_features_batch_masked(gpu_ctx.handle, C.byref(params), pyr.handle, n, 0, sel, buf.ctypes.data,
                                                             W - 1, 0, xx.ctypes.data, yy.ctypes.data,
                                                             vv.ctypes.data) == _capi.KLT_ERR_INVALID
    pyr.close()


# ---- sequences -------------------------------------------------------------------------------------------------------------
def sequence_frames(H, W, nframes, nseq, speed=5.0):
    from pyfeaturetrack_b200 import synth
    shifts = [(s[0] * speed, s[1] * speed) for s in synth.sequence_shifts(nframes)]
    return [synth.frames(H, W, shifts, seed=300 + s) for s in range(nseq)]


def oracle_masked_sequence(oracle, p, frames, n, mask_at):
    """The reference flow for one sequence (select, then per frame KLTTrackFeatures in sequentialMode + replacement on
    pyramid_last's level-0 gradients) with the selection of frame k restricted to mask_at(k) (None: no mask)."""
    state = {}
    pyr0 = oracle.image_pyramids(p, frames[0])
    x, y, v = masked_select(oracle, p, pyr0[1][0], pyr0[2][0], n, mask_at(0))
    state["pyramid_last"] = pyr0
    out = [(x.copy(), y.copy(), v.copy(), None)]
    for k in range(1, len(frames)):
        x, y, v, _ = oracle.track_features(p, frames[k - 1], frames[k], x, y, v, state)
        vt = v.copy()
        _, gxs, gys = state["pyramid_last"]
        x, y, v = masked_select(oracle, p, gxs[0], gys[0], n, mask_at(k), existing=(x, y, v))
        out.append((x.copy(), y.copy(), v.copy(), vt))
    return out


def run_masked_sequence(ctx, tc, seqs, n, masks_a, masks_b, change_at, off_at, wait=True):
    """Per-sequence masks masks_a from the start, masks_b (a host (B, H, W) array) from step change_at, none from off_at."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf, trackFeatures as tf
    B, nfr = len(seqs), len(seqs[0])
    H, W = seqs[0][0].shape
    q = _capi.Sequence(ctx, sgf.make_params(tc), tf._taps_for_one_image(tc), W, H, B, n, _capi.PRECISION_STRICT,
                       _capi.SELECT_STRICT)
    q.set_mask(np.stack(masks_a))
    q.start(np.ascontiguousarray(np.stack([s[0] for s in seqs])))
    out, graph_before_change, graph_after_change, pinned = [q.features()], None, None, []
    for k in range(1, nfr):
        if k == change_at:
            graph_before_change = q.uses_graph()
            q.set_mask(np.stack(masks_b))
        if k == off_at:
            q.set_mask(None)
        frames = np.ascontiguousarray(np.stack([s[k] for s in seqs]))
        if wait:
            q.step(frames)
            out.append(q.features())
        else:
            o = [ctx.pinned_array((B, n), np.float64), ctx.pinned_array((B, n), np.float64),
                 ctx.pinned_array((B, n), np.int32), ctx.pinned_array((B, n), np.int32)]
            q.step(frames, out=o)
            pinned.append(o)
        if k == off_at - 1:
            graph_after_change = q.uses_graph()
    q.sync()
    if not wait:
        out += [tuple(np.array(a) for a in o) for o in pinned]
        for o in pinned:
            for a in o:
                ctx.free_pinned(a)
    q.close()
    return out, graph_before_change, graph_after_change


@gpu
def test_sequence_masks_strict_equal_oracle(gpu_ctx, oracle, _quiet, monkeypatch):
    """STRICT + STRICT klt_sequence, 4 sequences x 15 frames, replacement, per-sequence masks: every list after every frame
    == the oracle sequence with the same masks.  The masks change at frame 8 while the steps replay from graphs (the graph
    replay stays on, the new masks apply from that step), and are turned off at frame 12 (the unmasked continuation).
    Enqueueing every step without waiting gives the same lists."""
    monkeypatch.delenv("KLT_B200_NO_GRAPH", raising=False)
    kw = dict(nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    tc, p = make_tc(**kw), oracle.Params(**kw)
    H, W, n, nfr, nseq = 480, 640, 300, 15, 4
    seqs = sequence_frames(H, W, nfr, nseq)
    masks_a = [make_mask(H, W, 100 + s) for s in range(nseq)]
    masks_b = [np.ascontiguousarray(np.roll(make_mask(H, W, 200 + s), 40, axis=1)) for s in range(nseq)]
    change_at, off_at = 8, 12
    got, g_before, g_after = run_masked_sequence(gpu_ctx, tc, seqs, n, masks_a, masks_b, change_at, off_at)
    assert g_before and g_after, "the steps were not replayed from CUDA graphs across the mask change"
    nowait, _, _ = run_masked_sequence(gpu_ctx, tc, seqs, n, masks_a, masks_b, change_at, off_at, wait=False)
    for k in range(nfr):
        for a, b in zip(got[k], nowait[k]):
            assert np.array_equal(a, b), k
    replaced = 0
    for s in range(nseq):
        def mask_at(k, s=s):
            return masks_a[s] if k < change_at else (masks_b[s] if k < off_at else None)
        want = oracle_masked_sequence(oracle, p, seqs[s], n, mask_at)
        for k in range(nfr):
            gx, gy, gv, gvt = got[k]
            eq((gx[s], gy[s], gv[s]), want[k][:3])
            if k:
                assert np.array_equal(gvt[s], want[k][3]), (s, k)
                new = (want[k][3] < 0) & (want[k][2] >= 0)
                replaced += int(new.sum())
                m = mask_at(k)
                if m is not None and new.any():
                    assert (m[want[k][1][new].astype(int), want[k][0][new].astype(int)] != 0).all()
    assert replaced > 20 * nseq


@gpu
def test_sequence_narrow_strip_widens_and_equals_composition(gpu_ctx, oracle, _quiet):
    """A 64-px allowed strip holds more candidates than the planned range but room for fewer features than slots: the walk
    widens its range (select_stats column 3 > 0) and the initial selection still == the composition; a device mask with an
    explicit pitch > w gives the same."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf, trackFeatures as tf
    kw = dict(nPyramidLevels=3, subsampling=2)
    tc, p = make_tc(**kw), oracle.Params(**kw)
    H, W, n, B = 480, 640, 400, 2
    frames = frames_for(H, W, B, 120)
    masks = []
    for b in range(B):
        m = np.zeros((H, W), np.uint8)
        m[:, 200 + 100 * b:264 + 100 * b] = 1
        masks.append(m)
    q = _capi.Sequence(gpu_ctx, sgf.make_params(tc), tf._taps_for_one_image(tc), W, H, B, n, _capi.PRECISION_STRICT,
                       _capi.SELECT_STRICT)
    q.set_mask(np.stack(masks))
    q.start(np.ascontiguousarray(np.stack(frames)))
    got = q.features()
    stats = q.select_stats()
    assert (stats[:, 3] > 0).all(), stats
    for b in range(B):
        _, gxs, gys = oracle.image_pyramids(p, frames[b])
        eq((got[0][b], got[1][b], got[2][b]), masked_select(oracle, p, gxs[0], gys[0], n, masks[b]))
        assert (got[2][b] >= 0).sum() < n
    buf, pitch, stride = lay_out(masks, W + 64, False)
    d = gpu_ctx.device_alloc(buf.nbytes)
    gpu_ctx.memcpy(d, buf, buf.nbytes)
    q.set_mask(d, pitch, stride)
    q.start(np.ascontiguousarray(np.stack(frames)))
    eq(q.features()[:3], got[:3])
    gpu_ctx.sync()
    gpu_ctx.device_free(d)
    with pytest.raises(ValueError):
        q.set_mask(np.ones((H, W + 1), np.uint8))
    q.close()


@gpu
def test_dropin_selection_mask(gpu_ctx, oracle, _quiet):
    """tc.selection_mask with KLTSelectGoodFeatures, KLTReplaceLostFeatures on a fresh selection pyramid and on
    tc.pyramid_last (sequentialMode) == the masked composition; a mask of the wrong shape is an error."""
    from pyfeaturetrack_b200 import config, synth, selectGoodFeatures as sgf, trackFeatures as tf
    config.set_precision(track="strict", select="strict")
    kw = dict(nPyramidLevels=3, subsampling=2)
    p = oracle.Params(**kw)
    H, W, n = 240, 320, 150
    f1, f2 = synth.frame_pair(H, W, seed=5)
    mask = make_mask(H, W, 55) != 0                  # a bool mask
    sm = oracle.smooth(f1.astype(np.float32), p.smooth_sigma(), p.cache)
    gx1, gy1 = oracle.gradients(sm, p.grad_sigma, p.cache)
    sm2 = oracle.smooth(f2.astype(np.float32), p.smooth_sigma(), p.cache)
    gx2, gy2 = oracle.gradients(sm2, p.grad_sigma, p.cache)
    for sequential in (False, True):
        tc = make_tc(sequentialMode=sequential, **kw)
        tc.selection_mask = mask
        fl = sgf.KLTSelectGoodFeatures(tc, f1, n)
        x, y, v = masked_select(oracle, p, gx1, gy1, n, mask)
        eq((np.array([float(f.x) for f in fl]), np.array([float(f.y) for f in fl]), np.array([f.val for f in fl], np.int32)),
           (x, y, v))
        if sequential:
            tf.KLTTrackFeatures(tc, f1, f2, fl)
            x, y, v, _ = oracle.track_features(p, f1, f2, x, y, v)
            _, gxs, gys = oracle.image_pyramids(p, f2)
            gx, gy = gxs[0], gys[0]
        else:
            gx, gy = gx2, gy2
        for i in range(0, n, 3):                      # lost slots to refill
            fl[i].val = -1
            fl[i].x = fl[i].y = -1
        x, y, v = knock_out(x, y, v)
        sgf.KLTReplaceLostFeatures(tc, f2, fl)
        want = masked_select(oracle, p, gx, gy, n, mask, existing=(x, y, v))
        eq((np.array([float(f.x) for f in fl]), np.array([float(f.y) for f in fl]), np.array([f.val for f in fl], np.int32)),
           want)
    tc = make_tc(**kw)
    tc.selection_mask = np.ones((H, W - 1), np.uint8)
    with pytest.raises(SystemExit):
        sgf.KLTSelectGoodFeatures(tc, f1, n)


@gpu
def test_no_mask_changes_no_launch_count(gpu_ctx, _quiet):
    """Without a mask a batched selection and a sequence step launch what they launched before the mask existed: the masked
    entry point with mask == NULL launches as many kernels as klt_select_good_features_batch, a mask adds exactly one
    (mask_premap), and a sequence step launches the same number of kernels never masked, masked, and after the mask is off."""
    from pyfeaturetrack_b200 import _capi, selectGoodFeatures as sgf, trackFeatures as tf
    H, W, B, n = 240, 320, 2, 100
    kw = dict(nPyramidLevels=2, subsampling=2, sequentialMode=True)
    tc = make_tc(**kw)
    frames = frames_for(H, W, B, 140)
    pyr = build_batch(gpu_ctx, tc, frames, _capi.PRECISION_STRICT)
    params = sgf.make_params(tc)
    x, y, v = np.full((B, n), -1.0), np.full((B, n), -1.0), np.full((B, n), -1, np.int32)
    mask = np.ones((H, W), np.uint8)

    def launches(fn):
        c0 = gpu_ctx.launch_count()
        fn()
        return gpu_ctx.launch_count() - c0
    for sel in (_capi.SELECT_STRICT, _capi.SELECT_FAST):
        for rep in (0, 1):
            plain = launches(lambda: gpu_ctx.check(_capi.lib().klt_select_good_features_batch(
                gpu_ctx.handle, C.byref(params), pyr.handle, n, rep, sel, x.ctypes.data, y.ctypes.data, v.ctypes.data)))
            null = launches(lambda: gpu_ctx.check(_capi.lib().klt_select_good_features_batch_masked(
                gpu_ctx.handle, C.byref(params), pyr.handle, n, rep, sel, None, 0, 0, x.ctypes.data, y.ctypes.data, v.ctypes.data)))
            masked = launches(lambda: gpu_ctx.check(_capi.lib().klt_select_good_features_batch_masked(
                gpu_ctx.handle, C.byref(params), pyr.handle, n, rep, sel, mask.ctypes.data, W, 0, x.ctypes.data, y.ctypes.data,
                v.ctypes.data)))
            assert plain == null and masked == plain + 1, (sel, rep, plain, null, masked)
    pyr.close()
    seq = sequence_frames(H, W, 12, B)
    per_step = {}
    for variant in ("never", "masked"):
        q = _capi.Sequence(gpu_ctx, params, tf._taps_for_one_image(tc), W, H, B, n, _capi.PRECISION_STRICT, _capi.SELECT_STRICT)
        q.start(np.ascontiguousarray(np.stack([s[0] for s in seq])))
        counts = []
        for k in range(1, 12):
            if variant == "masked" and k == 4:
                assert launches(lambda: q.set_mask(mask)) == 1
            if variant == "masked" and k == 8:
                assert launches(lambda: q.set_mask(None)) == 0
            counts.append(launches(lambda: q.step(np.ascontiguousarray(np.stack([s[k] for s in seq])))))
        q.sync()
        q.close()
        per_step[variant] = counts
    assert per_step["never"][-1] == per_step["never"][-2]
    assert per_step["masked"] == per_step["never"], per_step
