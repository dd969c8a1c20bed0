"""Drop-in for the reference's trackFeatures.py.  KLTTrackFeatures(tc, img1, img2, featurelist) keeps its
signature, mutates the feature list in place and returns None; pyramids and the Lucas-Kanade loop run on the GPU
(klt_pyr_build_u8 + klt_track_features)."""
from __future__ import print_function
import ctypes as C

import threading

import numpy as np

from . import _capi
from . import config
from . import convolve
from . import selectGoodFeatures as _sgf
from .klt import KLTCountRemainingFeatures, kltState, _fix_window
from .error import KLTError, KLTWarning
from .klt_util import KLTComputeSmoothSigma
from .pyramid import DevicePyramid
from .selectGoodFeatures import KLT_verbose, make_params, _image_size, _image_u8_or_f32


def _outOfBounds(x, y, ncols, nrows, borderx, bordery):
    return x < borderx or x > ncols - 1 - borderx or y < bordery or y > nrows - 1 - bordery


def _taps_for_one_image(tc):
    """Replays the kernel-cache lookups ComputeImagePyramids performs for ONE image (trackFeatures.py:165-172):
    smooth, then (L-1) pyramid smooths, then L gradient calls.  A stale-cache hit (convolve.py:236,258) therefore
    yields the same taps the reference would use."""
    taps = _capi.Taps()
    gauss, _ = convolve._kernels_for_smoothing(KLTComputeSmoothSigma(tc))
    taps.smooth = _capi.Kernel1D.from_taps(gauss)
    taps.pyramid = _capi.Kernel1D.from_taps([1.0])
    for _i in range(1, tc.nPyramidLevels):
        gauss, _ = convolve._kernels_for_smoothing(int(tc.subsampling) * tc.pyramid_sigma_fact)
        taps.pyramid = _capi.Kernel1D.from_taps(gauss)
    for _i in range(tc.nPyramidLevels):
        g, d = convolve._kernels_for_gradients(tc.grad_sigma)
    taps.grad_gauss, taps.grad_deriv = _capi.Kernel1D.from_taps(g), _capi.Kernel1D.from_taps(d)
    return taps


class _PyramidSet(object):
    """The three pyramids of one image on the device + the KLTPyramid-like views the reference API exposes."""

    def __init__(self, pyr):
        self.pyr = pyr
        self.img = DevicePyramid(pyr, 0)
        self.gradx = DevicePyramid(pyr, 1)
        self.grady = DevicePyramid(pyr, 2)


_hint = threading.local()     # .density = (features, pixels) of the KLTTrackFeatures call in progress on this thread:
                              # the input of config's `auto` mode


def _build_pyramids(tc, img, pyr):
    taps = _taps_for_one_image(tc)
    prec = config.track_precision_code(*(getattr(_hint, "density", None) or (None, None)))
    # stage through pinned memory: the upload becomes a true asynchronous DMA (it and the build overlap the host's work on
    # the next image); only enqueued here
    stage = _sgf._stage_u8(pyr.ctx, img, id(pyr))
    if stage is not None:
        pyr.build_u8(stage, taps, prec)
    else:
        a, _ = _image_u8_or_f32(img)
        pyr.build_f32(np.ascontiguousarray(a, np.float32), taps, prec, already_smoothed=False)
    return _PyramidSet(pyr)


@_capi.serialized
def ComputeImagePyramids(tc, img1, img2):
    """-> pyramid1, pyramid1_gradx, pyramid1_grady, pyramid2, pyramid2_gradx, pyramid2_grady (trackFeatures.py:146-196).
    The pyramids live on the device; `.img[i]` downloads a level on demand.  They are VIEWS of device memory this module
    recycles: outside sequentialMode the context's two scratch pyramids are rebuilt by the next call, in sequentialMode the
    pyramid of frame k-1 becomes the build target of frame k+1.  Copy the levels you want to keep (np.array(p.img[i]))
    before the next KLTTrackFeatures call; the reference returns independent arrays."""
    ctx = _capi.default_ctx()
    ncols, nrows = _image_size(img1)
    L, ss = int(tc.nPyramidLevels), int(float(tc.subsampling))
    if tc.sequentialMode and tc.pyramid_last is not None:
        pyramid1 = tc.pyramid_last
        if pyramid1.ncols[0] != ncols or pyramid1.nrows[0] != nrows:
            KLTError("(KLTTrackFeatures) Size of incoming image ({0} by {1}) is different from size of previous image ({2} by {3})".format(
                ncols, nrows, pyramid1.ncols[0], pyramid1.nrows[0]))
        assert tc.pyramid_last_gradx is not None
        assert tc.pyramid_last_grady is not None
        set1 = _PyramidSet.__new__(_PyramidSet)
        set1.pyr, set1.img, set1.gradx, set1.grady = pyramid1.pyr, pyramid1, tc.pyramid_last_gradx, tc.pyramid_last_grady
        # the second image must not overwrite the pyramid that is still in use
        pyr2 = _capi.Pyramid(ctx, ncols, nrows, L, ss, 1) if not hasattr(tc, "_klt_spare") or tc._klt_spare is None or \
            (tc._klt_spare.w, tc._klt_spare.h, tc._klt_spare.n_levels, tc._klt_spare.subsampling) != (ncols, nrows, L, ss) \
            else tc._klt_spare
    else:
        if tc.sequentialMode:
            pyr1 = _capi.Pyramid(ctx, ncols, nrows, L, ss, 1)
            pyr2 = _capi.Pyramid(ctx, ncols, nrows, L, ss, 1)
        else:
            pyr1 = ctx.scratch_pyramid(ncols, nrows, L, ss, 1, slot="track1")
            pyr2 = ctx.scratch_pyramid(ncols, nrows, L, ss, 1, slot="track2")
        set1 = _build_pyramids(tc, img1, pyr1)
    set2 = _build_pyramids(tc, img2, pyr2)
    return set1.img, set1.gradx, set1.grady, set2.img, set2.gradx, set2.grady


def _features_to_arrays(featurelist):
    n = len(featurelist)
    fl = _capi.featlist()
    if fl is not None and type(featurelist) is list:
        x, y, val = np.empty(n, np.float64), np.empty(n, np.float64), np.empty(n, np.int32)
        fl.klt_featlist_gather(featurelist, n, x.ctypes.data, y.ctypes.data, val.ctypes.data)
        return x, y, val
    val = np.fromiter((f.val for f in featurelist), np.int32, n)
    if n and val.min() >= 0:
        x = np.fromiter((f.x for f in featurelist), np.float64, n)
        y = np.fromiter((f.y for f in featurelist), np.float64, n)
    else:
        x = np.fromiter((f.x if f.val >= 0 else -1.0 for f in featurelist), np.float64, n)
        y = np.fromiter((f.y if f.val >= 0 else -1.0 for f in featurelist), np.float64, n)
    return x, y, val


class AffineTemplate(object):
    """feat.aff_img / aff_img_gradx / aff_img_grady: the (aw+2) x (ah+2) template kept on the device; converts to a
    NumPy array on demand (np.asarray(feat.aff_img)) and pickles as that array."""

    def __init__(self, state, slot, which):
        self.state, self.slot, self.which = state, slot, which

    def __array__(self, dtype=None, copy=None):
        a = self.state.template(self.slot)[self.which]
        return a if dtype is None else a.astype(dtype)

    def __reduce__(self):
        return (np.array, (self.__array__(),))


def _affine_state(tc, ctx, featurelist):
    """The klt_affine of this tracking context, with the slots of features that carry no template reset
    (freshly selected or replaced features have aff_img = None, selectGoodFeatures.py:120-128)."""
    n = len(featurelist)
    st = getattr(tc, "_klt_affine", None)
    if st is None or st.n != n or st.aw != tc.affine_window_width or st.ah != tc.affine_window_height or st.ctx is not ctx:
        st = tc._klt_affine = _capi.AffineState(ctx, n, int(tc.affine_window_width), int(tc.affine_window_height))
    # slots whose feature does not carry this state's template (fresh, replaced or foreign features) start over
    keep = [type(t) is AffineTemplate and t.state is st and t.slot == i
            for i, t in enumerate([f.__dict__.get("aff_img") for f in featurelist])]
    if not all(keep):
        st.reset(np.logical_not(np.array(keep, dtype=bool)).astype(np.int32))
    return st


def _clear_affine(feat):
    feat.aff_img = None
    feat.aff_img_gradx = None
    feat.aff_img_grady = None


@_capi.serialized
def KLTTrackFeatures(tc, img1, img2, featurelist):
    assert _image_size(img1) == _image_size(img2)
    ncols, nrows = _image_size(img1)
    if KLT_verbose >= 1:
        print("(KLT) Tracking {0} features in a {1} by {2} image...  ".format(
            KLTCountRemainingFeatures(featurelist), ncols, nrows))
    _fix_window(tc, "Tracking context")
    use_affine = tc.affineConsistencyCheck >= 0
    max_fb_error = getattr(tc, "max_fb_error", None)
    if (tc.lighting_insensitive or max_fb_error is not None) and use_affine:
        # the reference raises for lighting_insensitive alone (trackFeaturesUtils.pyx:435); this build implements the
        # mode from the C the reference carries as comments (:152-239) -- but not together with the affine check, and
        # neither is the forward-backward check (beyond the reference)
        raise Exception("Not implemented")
    if use_affine and tc.affineConsistencyCheck > 2:
        raise ValueError("affineConsistencyCheck must be -1, 0, 1 or 2")

    # the affine block reads gradient planes, so `auto` should build them in the fused dense pass right away
    _hint.density = (len(featurelist) if not use_affine else 1 << 60, ncols * nrows)
    try:
        pyramid1, pyramid1_gradx, pyramid1_grady, pyramid2, pyramid2_gradx, pyramid2_grady = ComputeImagePyramids(tc, img1, img2)
    finally:
        _hint.density = None
    ctx = pyramid1.pyr.ctx
    if tc.writeInternalImages:
        # trackFeatures.py:186-196 (the reference's own dump dies on ndarray.save; this writes the files it names)
        from .klt_util import KLTWriteFloatImageToPGM
        for i in range(int(tc.nPyramidLevels)):
            for tag, p, gx, gy in (("i", pyramid1, pyramid1_gradx, pyramid1_grady), ("j", pyramid2, pyramid2_gradx, pyramid2_grady)):
                KLTWriteFloatImageToPGM(p.img[i], "kltimg_tf_{0}{1}.pgm".format(tag, i))
                KLTWriteFloatImageToPGM(gx.img[i], "kltimg_tf_{0}{1}_gx.pgm".format(tag, i))
                KLTWriteFloatImageToPGM(gy.img[i], "kltimg_tf_{0}{1}_gy.pgm".format(tag, i))
    x, y, val = _features_to_arrays(featurelist)
    was_live = val >= 0
    old_val = val.copy()
    params = make_params(tc)
    aff = None
    if use_affine:
        # The reference's affine block (trackFeatures.py:347-399) calls three undefined functions; this runs the C-KLT
        # routines of those names on the GPU.  Per-feature state lives in a klt_affine keyed by list position.
        aff = _affine_state(tc, ctx, featurelist)
        ctx.check(_capi.lib().klt_track_features_affine(ctx.handle, C.byref(params), pyramid1.pyr.handle,
                                                       pyramid2.pyr.handle, len(featurelist), x.ctypes.data,
                                                       y.ctypes.data, val.ctypes.data, aff.handle, None))
    elif max_fb_error is not None:
        # forward-backward check: rejected features come back with val = kltState.KLT_FB_ERROR
        ctx.check(_capi.lib().klt_track_features_fb(ctx.handle, C.byref(params), pyramid1.pyr.handle, pyramid2.pyr.handle,
                                                   len(featurelist), float(max_fb_error), x.ctypes.data, y.ctypes.data,
                                                   val.ctypes.data, None, None))
    else:
        ctx.check(_capi.lib().klt_track_features(ctx.handle, C.byref(params), pyramid1.pyr.handle, pyramid2.pyr.handle,
                                                len(featurelist), x.ctypes.data, y.ctypes.data, val.ctypes.data, None))
    ctx.mark_synced()          # host arrays: the tracking call waited for the stream
    fl = _capi.featlist()
    if fl is not None and type(featurelist) is list:
        fl.klt_featlist_scatter_tracked(featurelist, len(featurelist), x.ctypes.data, y.ctypes.data, val.ctypes.data,
                                        old_val.ctypes.data)
    else:
        xs, ys, vals = x.tolist(), y.tolist(), val.tolist()
        for feat, live, fx, fy, v in zip(featurelist, was_live.tolist(), xs, ys, vals):
            if not live:
                continue                                             # trackFeatures.py:253
            d = feat.__dict__
            if v == 0:                                               # KLT_TRACKED
                d["x"] = fx; d["y"] = fy; d["val"] = 0
            else:
                d["x"] = -1.0; d["y"] = -1.0; d["val"] = v
                if "aff_img" in d:
                    _clear_affine(feat)

    if use_affine:
        has, ax, ay, A = aff.download()
        rows = zip(featurelist, was_live.tolist(), has.tolist(), ax.astype(np.float64).tolist(), ay.astype(np.float64).tolist(),
                   A.astype(np.float64).tolist())
        for i, (feat, live, h, fax, fay, fA) in enumerate(rows):
            if not live:
                continue
            d = feat.__dict__
            d["aff_x"] = fax; d["aff_y"] = fay
            d["aff_Axx"], d["aff_Ayx"], d["aff_Axy"], d["aff_Ayy"] = fA
            if h:
                if type(d.get("aff_img")) is not AffineTemplate:
                    d["aff_img"], d["aff_img_gradx"], d["aff_img_grady"] = (AffineTemplate(aff, i, w) for w in range(3))
            else:
                d["aff_img"] = d["aff_img_gradx"] = d["aff_img_grady"] = None

    if tc.sequentialMode:
        if tc.pyramid_last is not None and tc.pyramid_last is not pyramid2:
            tc._klt_spare = tc.pyramid_last.pyr                  # recycle the older pyramid's device memory
        tc.pyramid_last = pyramid2
        tc.pyramid_last_gradx = pyramid2_gradx
        tc.pyramid_last_grady = pyramid2_grady

    if KLT_verbose >= 1:
        print("\n\t{0} features successfully tracked.".format(KLTCountRemainingFeatures(featurelist)))
        if tc.writeInternalImages:
            print("\tWrote images to 'kltimg_tf*.pgm'.")
