"""Drop-in for the reference's selectGoodFeatures.py.  KLTSelectGoodFeatures(tc, img, nFeatures) keeps its
signature and return convention (a fresh list of KLT_Feature); the work -- smoothing, gradients, summed-area
tables, min-eigenvalue map, descending sort and greedy minimum-distance suppression -- runs on the GPU
(klt_pyr_build_u8 + klt_select_good_features)."""
from __future__ import print_function
import ctypes as C

import numpy as np

from . import _capi
from . import config
from . import convolve
from .klt import KLT_Feature, KLTCountRemainingFeatures, kltState, _fix_window
from .error import KLTError, KLTWarning
from .klt_util import KLTComputeSmoothSigma


class selectionMode:
    SELECTING_ALL = 1
    REPLACING_SOME = 2


KLT_verbose = 1


def _image_size(img):
    if isinstance(img, np.ndarray):
        return img.shape[1], img.shape[0]
    return img.size


def _image_u8_or_f32(img):
    """PIL 'L' images and uint8 arrays go to the GPU as bytes (img.convert("F") is exact for them);
    anything else is converted to float32 the way the reference does (selectGoodFeatures.py:190)."""
    if isinstance(img, np.ndarray):
        a = img
    elif getattr(img, "mode", None) == "L":
        a = np.asarray(img)
    else:
        a = np.asarray(img.convert("F"))
    if a.dtype == np.uint8:
        return np.ascontiguousarray(a), True
    return np.ascontiguousarray(a, np.float32), False


def _pil_into(stage, img, w, h):
    """Pixels of a PIL 'L' image -> the uint8 array `stage` in ONE pass: PIL's core paste into an image that maps the array's
    memory (Image.frombuffer); where that private path is not available, the raw encoder in 64-row chunks (its output
    buffer then stays a small reused heap block instead of a fresh 2 MB mmap per image) and a memmove per chunk.
    Measured per 1080p image on the bench host: np.asarray 0.47 ms, one encode 0.29, chunks 0.22, paste ~0.1."""
    from PIL import Image
    img.load()
    try:
        view = _pil_views.get(stage.ctypes.data)
        if view is None or view[0] is not stage:
            if len(_pil_views) > 16:
                _pil_views.clear()
            view = _pil_views[stage.ctypes.data] = (stage, Image.frombuffer("L", (w, h), stage, "raw", "L", 0, 1))
        view[1].im.paste(img.im, (0, 0, w, h))
        return
    except Exception:
        pass
    enc = Image._getencoder("L", "raw", ("L",))
    try:
        enc.setimage(img.im)
    except TypeError:
        enc.setimage(img.im, (0, 0) + img.size)
    base, off, chunk, total = stage.ctypes.data, 0, max(w * 64, 65536), w * h
    while True:
        _, err, data = enc.encode(chunk)
        if off + len(data) > total:
            raise ValueError("long read")
        C.memmove(base + off, data, len(data))
        off += len(data)
        if err:
            break
    if err < 0 or off != total:
        raise ValueError("short read")


_pil_views = {}     # staging array address -> (array, PIL image mapping its memory)


def _stage_u8(ctx, img, key):
    """The image as uint8 [h, w] in a pinned staging buffer of `ctx` (one per key), ready for an asynchronous upload; None if the
    image is not 8-bit (the caller converts to float32 like the reference).  PIL 'L' images are written into the pinned buffer
    directly (_pil_into); any surprise from PIL's private API falls back to np.asarray."""
    if isinstance(img, np.ndarray):
        if img.dtype != np.uint8 or img.ndim != 2:
            return None
        stage = ctx.pinned_stage(img.shape, key)
        ctx.sync_stage(key)
        np.copyto(stage, img)
        return stage
    if getattr(img, "mode", None) != "L":
        return None
    w, h = img.size
    stage = ctx.pinned_stage((h, w), key)
    ctx.sync_stage(key)
    try:
        _pil_into(stage, img, w, h)
    except Exception:
        np.copyto(stage, np.asarray(img))
    return stage


def make_params(tc):
    p = _capi.Params()
    p.window_width, p.window_height = int(tc.window_width), int(tc.window_height)
    p.n_levels, p.subsampling = int(tc.nPyramidLevels), int(tc.subsampling)
    p.borderx, p.bordery = float(tc.borderx), float(tc.bordery)
    p.mindist, p.min_eigenvalue = int(tc.mindist), int(tc.min_eigenvalue)
    if tc.min_eigenvalue != int(tc.min_eigenvalue):
        # val >= tc.min_eigenvalue is a float32-vs-Python-float comparison in the reference (selectGoodFeatures.py:116): for a
        # float32 val it equals val >= (the smallest float32 that is >= the Python value)
        m = np.float32(tc.min_eigenvalue)
        if float(m) < float(tc.min_eigenvalue):
            m = np.nextafter(m, np.float32(np.inf))
        p.min_eigenvalue_f = float(m)
    p.n_skipped_pixels = int(tc.nSkippedPixels)
    p.max_iterations = int(tc.max_iterations)
    p.min_determinant, p.min_displacement, p.step_factor = tc.min_determinant, tc.min_displacement, tc.step_factor
    p.has_max_residue = 0 if tc.max_residue is None else 1
    p.max_residue = 0.0 if tc.max_residue is None else tc.max_residue
    p.retain_trackers = 1 if tc.retainTrackers else 0
    p.lighting_insensitive = 1 if tc.lighting_insensitive else 0
    p.affine_consistency_check = int(tc.affineConsistencyCheck)
    p.affine_window_width, p.affine_window_height = int(tc.affine_window_width), int(tc.affine_window_height)
    p.affine_max_iterations = int(tc.affine_max_iterations)
    p.affine_max_residue = tc.affine_max_residue
    p.affine_min_displacement = tc.affine_min_displacement
    p.affine_max_displacement_differ = tc.affine_max_displacement_differ
    return p


# attributes a (re)selected feature starts with (selectGoodFeatures.py:120-128)
_AFFINE_RESET = dict(aff_img=None, aff_img_gradx=None, aff_img_grady=None, aff_x=-1.0, aff_y=-1.0, aff_Axx=1.0,
                     aff_Ayx=0.0, aff_Axy=0.0, aff_Ayy=1.0)


def _selection_mask(tc, ncols, nrows):
    """tc.selection_mask as uint8 [nrows, ncols] (nonzero = new features allowed there), or None."""
    m = getattr(tc, "selection_mask", None)
    if m is None:
        return None
    m = np.asarray(m)
    if m.shape != (nrows, ncols):
        KLTError("(_KLTSelectGoodFeatures) Size of tc.selection_mask ({0}) is different from size of image ({1} by {2})".format(
            " by ".join(str(s) for s in m.shape[::-1]), ncols, nrows))
    return np.ascontiguousarray(m != 0, np.uint8)


def _select_on_device(tc, pyr, nFeatures, featurelist, overwriteAllFeatures):
    """Scan + sort + _enforceMinimumDistance on level-0 gradients of `pyr` (selectGoodFeatures.py:215-246), restricted to
    tc.selection_mask where one is set (beyond the reference)."""
    ctx = pyr.ctx
    mask = _selection_mask(tc, pyr.w, pyr.h)
    x, y, val = _gather(featurelist, nFeatures, overwriteAllFeatures)
    old_val = val.copy()
    params = make_params(tc)
    if mask is None:
        ctx.check(_capi.lib().klt_select_good_features_batch(ctx.handle, C.byref(params), pyr.handle, nFeatures,
                                                            0 if overwriteAllFeatures else 1, config.select_mode_code(),
                                                            x.ctypes.data, y.ctypes.data, val.ctypes.data))
    else:
        ctx.check(_capi.lib().klt_select_good_features_batch_masked(ctx.handle, C.byref(params), pyr.handle, nFeatures,
                                                                   0 if overwriteAllFeatures else 1, config.select_mode_code(),
                                                                   mask.ctypes.data, pyr.w, 0, x.ctypes.data, y.ctypes.data,
                                                                   val.ctypes.data))
    ctx.mark_synced()          # host arrays: the call waited for the stream
    _scatter(featurelist, x, y, val, old_val, overwriteAllFeatures)
    return featurelist


def _gather(featurelist, n, overwriteAllFeatures):
    """x, y, val arrays of the list for the C ABI (all -1 / KLT_NOT_FOUND when every slot is overwritten)."""
    if overwriteAllFeatures:
        return np.full(n, -1.0), np.full(n, -1.0), np.full(n, kltState.KLT_NOT_FOUND, np.int32)
    return (np.fromiter((f.x for f in featurelist), np.float64, n), np.fromiter((f.y for f in featurelist), np.float64, n),
            np.fromiter((f.val for f in featurelist), np.int32, n))


def _scatter(featurelist, x, y, val, old_val, overwriteAllFeatures):
    """Write the selection back into the KLT_Feature objects (selectGoodFeatures.py:110-128): x, y become np.int32 and
    val a Python int (quirk Q13); lists instead of per-element ndarray indexing keep this loop off the profile."""
    xi, yi, vi = list(x.astype(np.int32)), list(y.astype(np.int32)), val.tolist()
    if overwriteAllFeatures:
        for feat, xv, yv, v in zip(featurelist, xi, yi, vi):
            d = feat.__dict__
            if v >= 0:
                d["x"], d["y"], d["val"] = xv, yv, v
            else:
                d["x"], d["y"], d["val"] = -1, -1, kltState.KLT_NOT_FOUND    # C-KLT's fill (quirk Q6)
            d.update(_AFFINE_RESET)
    else:
        for i in np.flatnonzero((old_val < 0) & (val >= 0)).tolist():
            d = featurelist[i].__dict__
            d["x"], d["y"], d["val"] = xi[i], yi[i], vi[i]
            d.update(_AFFINE_RESET)


@_capi.serialized
def _enforceMinimumDistance(pointlist, featurelist, ncols, nrows, mindist, min_eigenvalue, overwriteAllFeatures):
    """Greedy minimum-distance suppression over a caller-ordered list of (val, x, y) tuples (selectGoodFeatures.py:45-135),
    on the GPU (klt_enforce_min_distance).  Mutates and returns featurelist."""
    ctx = _capi.default_ctx()
    n = len(featurelist)
    x, y, val = _gather(featurelist, n, overwriteAllFeatures)
    old_val = val.copy()
    pv = np.ascontiguousarray([p[0] for p in pointlist], np.float32)
    px = np.ascontiguousarray([p[1] for p in pointlist], np.int32)
    py = np.ascontiguousarray([p[2] for p in pointlist], np.int32)
    ctx.check(_capi.lib().klt_enforce_min_distance(ctx.handle, len(pointlist), pv.ctypes.data, px.ctypes.data, py.ctypes.data,
                                                  int(ncols), int(nrows), int(mindist), float(min_eigenvalue),
                                                  1 if overwriteAllFeatures else 0, n, x.ctypes.data, y.ctypes.data,
                                                  val.ctypes.data))
    _scatter(featurelist, x, y, val, old_val, overwriteAllFeatures)
    return featurelist


def _selection_pyramid(tc, img):
    """float image -> (optional) smooth -> gradients, as a 1-level device pyramid (selectGoodFeatures.py:181-197)."""
    ctx = _capi.default_ctx()
    ncols, nrows = _image_size(img)
    a = _stage_u8(ctx, img, "select") if tc.smoothBeforeSelecting else None
    is_u8 = a is not None
    if not is_u8:
        a, is_u8 = _image_u8_or_f32(img)
    taps = _capi.Taps()
    one = _capi.Kernel1D.from_taps([1.0])
    taps.pyramid = one
    if tc.smoothBeforeSelecting:
        gauss, _ = convolve._kernels_for_smoothing(KLTComputeSmoothSigma(tc))
        taps.smooth = _capi.Kernel1D.from_taps(gauss)
    else:
        taps.smooth = one
    g, d = convolve._kernels_for_gradients(tc.grad_sigma)
    taps.grad_gauss, taps.grad_deriv = _capi.Kernel1D.from_taps(g), _capi.Kernel1D.from_taps(d)
    pyr = ctx.scratch_pyramid(ncols, nrows, 1, 2, 1, slot="select")
    prec = config.select_precision_code()
    if tc.smoothBeforeSelecting:
        if is_u8:
            pyr.build_u8(a, taps, prec)
        else:
            pyr.build_f32(a, taps, prec, already_smoothed=False)
    else:
        pyr.build_f32(np.ascontiguousarray(a, np.float32), taps, prec, already_smoothed=True)
    return pyr


@_capi.serialized
def _KLTSelectGoodFeatures(tc, img, nFeatures, mode, featurelist=None):
    overwriteAllFeatures = (mode == selectionMode.SELECTING_ALL)
    if featurelist is None:
        featurelist = [KLT_Feature() for i in range(nFeatures)]
    _fix_window(tc, "Tracking context")
    if mode == selectionMode.REPLACING_SOME and tc.sequentialMode and tc.pyramid_last is not None:
        pyr = tc.pyramid_last.pyr          # level-0 gradients of the last tracked image (selectGoodFeatures.py:176-179)
    else:
        pyr = _selection_pyramid(tc, img)
    if tc.writeInternalImages:
        # selectGoodFeatures.py:201-204 (the reference's own dump dies on ndarray.save; this writes the files it names)
        from .klt_util import KLTWriteFloatImageToPGM
        for which, name in ((0, "kltimg_sgfrlf.pgm"), (1, "kltimg_sgfrlf_gx.pgm"), (2, "kltimg_sgfrlf_gy.pgm")):
            KLTWriteFloatImageToPGM(pyr.download(which, 0), name)
    if tc.mindist < 0:
        KLTWarning("(_KLTSelectGoodFeatures) Tracking context field tc.mindist is negative ({0}); setting to zero".format(tc.mindist))
        tc.mindist = 0
    return _select_on_device(tc, pyr, len(featurelist), featurelist, overwriteAllFeatures)


def KLTSelectGoodFeatures(tc, img, nFeatures):
    ncols, nrows = _image_size(img)
    if KLT_verbose >= 1:
        print("(KLT) Selecting the {0} best features from a {1} by {2} image...  ".format(nFeatures, ncols, nrows))
    fl = _KLTSelectGoodFeatures(tc, img, nFeatures, selectionMode.SELECTING_ALL)
    if KLT_verbose >= 1:
        print("\n\t{0} features found.\n".format(KLTCountRemainingFeatures(fl)))
        if tc.writeInternalImages:
            print("\tWrote images to 'kltimg_sgfrlf*.pgm'.\n")
    return fl


def KLTReplaceLostFeatures(tc, img, fl):
    """C-KLT's KLTReplaceLostFeatures: refill the slots of lost features (val < 0) with the best new features that
    keep mindist from the survivors.  The reference has only the mode constant (selectGoodFeatures.py:11-13) and
    _enforceMinimumDistance(..., overwriteAllFeatures=False), which this follows."""
    nLost = len(fl) - KLTCountRemainingFeatures(fl)
    ncols, nrows = _image_size(img)
    if KLT_verbose >= 1:
        print("(KLT) Attempting to replace {0} features in a {1} by {2} image...  ".format(nLost, ncols, nrows))
    if nLost > 0:
        _KLTSelectGoodFeatures(tc, img, len(fl), selectionMode.REPLACING_SOME, fl)
    if KLT_verbose >= 1:
        print("\n\t{0} features replaced.".format(nLost - len(fl) + KLTCountRemainingFeatures(fl)))
