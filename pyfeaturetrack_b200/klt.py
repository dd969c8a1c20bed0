"""Drop-in for the reference's klt.py: tracking context, feature type, status codes (klt.py:23-325).
Pure host-side Python, same field names and defaults; border math keeps Python-3 true division (quirk Q1)."""
from __future__ import print_function
import math

from .error import KLTError, KLTWarning
from .convolve import KLTGetKernelWidths
from .klt_util import KLTComputeSmoothSigma


class kltState:
    KLT_TRACKED = 0
    KLT_NOT_FOUND = -1
    KLT_SMALL_DET = -2
    KLT_MAX_ITERATIONS = -3
    KLT_OOB = -4
    KLT_LARGE_RESIDUE = -5
    KLT_FB_ERROR = -6            # beyond the reference: rejected by the forward-backward check (tc.max_fb_error)


def _fix_window(tc, who):
    """Odd, >= 3 window (klt.py:86-102,142-158); mutates tc and warns like the reference."""
    if tc.window_width % 2 != 1:
        tc.window_width = tc.window_width + 1
        KLTWarning("({0}) Window width must be odd.  Changing to {1}.\n".format(who, tc.window_width))
    if tc.window_height % 2 != 1:
        tc.window_height = tc.window_height + 1
        KLTWarning("({0}) Window height must be odd.  Changing to {1}.\n".format(who, tc.window_height))
    if tc.window_width < 3:
        tc.window_width = 3
        KLTWarning("({0}) Window width must be at least three.  \nChanging to {1}.\n".format(who, tc.window_width))
    if tc.window_height < 3:
        tc.window_height = 3
        KLTWarning("({0}) Window height must be at least three.  \nChanging to {1}.\n".format(who, tc.window_height))


# field -> default (klt.py:45-73 of the reference; documented there at :200-246)
_TC_DEFAULTS = (
    ("mindist", 10), ("window_width", 7), ("window_height", 7),
    ("sequentialMode", False), ("retainTrackers", False), ("smoothBeforeSelecting", True),
    ("writeInternalImages", False), ("lighting_insensitive", False),
    ("min_eigenvalue", 1), ("min_determinant", 0.01), ("max_iterations", 10), ("min_displacement", 0.1),
    ("max_residue", None),                       # None switches the residue check off (quirk Q4)
    ("grad_sigma", 1.0), ("smooth_sigma_fact", 0.1), ("pyramid_sigma_fact", 0.9), ("step_factor", 1.0),
    ("nSkippedPixels", 0),
    ("pyramid_last", None), ("pyramid_last_gradx", None), ("pyramid_last_grady", None),
    # affine consistency check
    ("affineConsistencyCheck", -1), ("affine_window_width", 15), ("affine_window_height", 15),
    ("affine_max_iterations", 10), ("affine_max_residue", 10.), ("affine_min_displacement", 0.02),
    ("affine_max_displacement_differ", 1.5),
    # beyond the reference: forward-backward check (level-0 pixels); None switches it off
    ("max_fb_error", None),
)
# search_range / window_halfwidth <= bound  ->  (nPyramidLevels, subsampling)   (klt.py:105-117)
_PYRAMID_STEPS = ((3.0, 2, 2), (5.0, 2, 4), (9.0, 2, 8))


class KLT_TrackingContext:
    def __init__(self):
        for name, value in _TC_DEFAULTS:
            setattr(self, name, value)
        self.KLTChangeTCPyramid(15)          # klt.py:76-77: search range 15 -> 2 levels, subsampling 4 for 7x7
        self.KLTUpdateTCBorder()

    def KLTChangeTCPyramid(self, search_range):
        """Pyramid depth / subsampling heuristic (klt.py:84-128)."""
        _fix_window(self, "KLTChangeTCPyramid")
        ratio = float(search_range) / (min(self.window_width, self.window_height) / 2.0)
        if ratio < 1.0:
            self.nPyramidLevels = 1          # subsampling keeps its previous value (quirk Q12)
            return
        for bound, levels, ss in _PYRAMID_STEPS:
            if ratio <= bound:
                self.nPyramidLevels, self.subsampling = levels, ss
                return
        # search_range = halfwidth * (8^levels - 1) / 7, rounded up
        self.nPyramidLevels = int(float(math.log(7.0 * ratio + 1.0) / math.log(8.0)) + 0.99)
        self.subsampling = 8

    def KLTUpdateTCBorder(self):
        """Border lost to convolution and windows (klt.py:137-189)."""
        num_levels = self.nPyramidLevels
        ss = self.subsampling
        _fix_window(self, "KLTUpdateTCBorder")
        window_hw = max(self.window_width, self.window_height) / 2
        gauss_width, gaussderiv_width = KLTGetKernelWidths(KLTComputeSmoothSigma(self))
        smooth_gauss_hw = gauss_width / 2
        gauss_width, gaussderiv_width = KLTGetKernelWidths(_pyramidSigma(self))
        pyramid_gauss_hw = gauss_width / 2
        n_invalid_pixels = smooth_gauss_hw
        for i in range(1, num_levels):
            val = (float(n_invalid_pixels) + pyramid_gauss_hw) / ss
            n_invalid_pixels = int(val + 0.99)
        ss_power = 1
        for i in range(1, num_levels):
            ss_power *= ss
        border = (n_invalid_pixels + window_hw) * ss_power
        self.borderx = border
        self.bordery = border

    def __getstate__(self):
        # device-resident pyramids cannot be pickled; sequential state restarts after unpickling
        d = dict((k, v) for k, v in self.__dict__.items() if not k.startswith("_klt"))
        d["pyramid_last"] = d["pyramid_last_gradx"] = d["pyramid_last_grady"] = None
        return d


def _pyramidSigma(tc):
    return (tc.pyramid_sigma_fact * tc.subsampling)


class KLT_Feature:
    """Attributes appear when assigned, exactly like the reference's class (klt.py:249-263, quirk Q5)."""

    def __init__(self):
        pass


class KLT_FeatureHistory:
    pass


class KLT_FeatureTable:
    pass


def KLTPrintTrackingContext(tc):
    print(tc)
    print("\n\nTracking context:\n")
    for name in ("mindist", "window_width", "window_height", "sequentialMode", "smoothBeforeSelecting",
                 "writeInternalImages"):
        print("\t{0} = {1}".format(name, getattr(tc, name)))
    for name in ("min_eigenvalue", "min_determinant", "min_displacement", "max_iterations", "max_residue",
                 "grad_sigma", "smooth_sigma_fact", "pyramid_sigma_fact", "nSkippedPixels", "borderx", "bordery",
                 "nPyramidLevels", "subsampling"):
        print("\t{0} = {1}".format(name, getattr(tc, name)))
    print("\n\tpyramid_last = {0}".format(tc.pyramid_last))
    print("\tpyramid_last_gradx = {0}".format(tc.pyramid_last_gradx))
    print("\tpyramid_last_grady = {0}".format(tc.pyramid_last_grady))
    print("\n")


def KLTCountRemainingFeatures(fl):
    count = 0
    for feat in fl:
        if feat.val >= 0:
            count = count + 1
    return count
