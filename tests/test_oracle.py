"""CPU tests: the oracle (oracle/klt_oracle.c) against the golden vectors produced by the unmodified reference
(tests/golden/make_golden.py) and, when oracle/_ref is present, against the reference itself run live."""
import numpy as np
import pytest


def P(oracle, **kw):
    return oracle.Params(**kw)


def fl(golden, key):
    a = golden[key]
    return a[0], a[1], a[2].astype(np.int32)


def assert_features_equal(got, want):
    gx, gy, gv = got
    wx, wy, wv = want
    assert np.array_equal(np.asarray(gv, np.int64), np.asarray(wv, np.int64))
    assert np.array_equal(np.asarray(gx, np.float64), np.asarray(wx, np.float64))
    assert np.array_equal(np.asarray(gy, np.float64), np.asarray(wy, np.float64))


@pytest.mark.parametrize("sigma", [0.7, 1.0, 1.5, 1.8, 3.6, 7.2])
def test_kernel_taps_bit_exact(oracle, golden, sigma):
    g, d = oracle.compute_kernels(sigma)
    assert np.array_equal(g, golden["taps_g_%s" % sigma])
    assert np.array_equal(d, golden["taps_d_%s" % sigma])


def test_kernel_too_wide(oracle):
    with pytest.raises(oracle.KernelTooWide):
        oracle.compute_kernels(14.4)


def test_borders(oracle, golden):
    for w, L, ss, border in golden["borders"]:
        p = P(oracle, window_width=int(w), window_height=int(w), nPyramidLevels=int(L), subsampling=int(ss))
        assert p.borderx == border


def test_images_bit_exact(oracle, golden, img01):
    p = P(oracle)
    f0 = img01[0].astype(np.float32)
    sm = oracle.smooth(f0, 0.7, p.cache)
    assert np.array_equal(sm, golden["A_smooth"])
    gx, gy = oracle.gradients(sm, 1.0, p.cache)
    assert np.array_equal(gx, golden["A_gradx"])
    assert np.array_equal(gy, golden["A_grady"])
    pyr = oracle.pyramid(sm, 4, 2, 0.9, p.cache)
    assert np.array_equal(pyr[1], golden["A_pyr1"])
    g1x, g1y = oracle.gradients(pyr[1], 1.0, p.cache)
    assert np.array_equal(g1x, golden["A_pyr1_gradx"])
    assert np.array_equal(g1y, golden["A_pyr1_grady"])


def test_scan_bit_exact(oracle, golden):
    val, xs, ys = oracle.scan_good_features(golden["A_gradx"], golden["A_grady"], 30, 30, 3, 3, 0)
    assert np.array_equal(val, golden["A_scan_val"])
    assert xs[0] == 30 and ys[0] == 30


def test_patch_bit_exact(oracle, golden):
    assert np.array_equal(oracle.extract_patch(golden["A_smooth"], 100.3, 57.8, 7, 7), golden["A_patch"])
    with pytest.raises(AssertionError):
        oracle.extract_patch(golden["A_smooth"], 2.5, 57.8, 7, 7)


@pytest.mark.parametrize("n", [50, 100])
def test_config_A_select_and_track(oracle, golden, img01, n):
    p = P(oracle, max_residue=10.0)
    sel = oracle.select_good_features(p, img01[0], n)
    assert_features_equal(sel, fl(golden, "A_sel%d" % n))
    trk = oracle.track_features(p, img01[0], img01[1], *sel)[:3]
    assert_features_equal(trk, fl(golden, "A_trk%d" % n))
    back = oracle.track_features(p, img01[1], img01[0], *trk)[:3]
    assert_features_equal(back, fl(golden, "A_trk%d_back" % n))


def test_config_A_variants(oracle, golden, img01):
    p = P(oracle)
    sel = oracle.select_good_features(p, img01[0], 60)
    assert_features_equal(oracle.track_features(p, img01[0], img01[1], *sel)[:3], fl(golden, "A_trk60_nores"))
    p = P(oracle, retainTrackers=True)
    sel = oracle.select_good_features(p, img01[0], 60)
    assert_features_equal(oracle.track_features(p, img01[0], img01[1], *sel)[:3], fl(golden, "A_trk60_retain"))
    p = P(oracle, nSkippedPixels=2, mindist=15, min_eigenvalue=500)
    assert_features_equal(oracle.select_good_features(p, img01[0], 40), fl(golden, "A_sel40_skip2"))
    p = P(oracle, smoothBeforeSelecting=False)
    assert_features_equal(oracle.select_good_features(p, img01[0], 40), fl(golden, "A_sel40_nosmooth"))


def test_sequential_with_replacement(oracle, golden, img01):
    p = P(oracle, max_residue=10.0, sequentialMode=True)
    x, y, v = oracle.select_good_features(p, img01[0], 80)
    state = {}
    want = golden["A_seq80"]
    k = 0
    for a, b in ((0, 1), (1, 0), (0, 1)):
        x, y, v, _ = oracle.track_features(p, img01[a], img01[b], x, y, v, state)
        assert_features_equal((x, y, v), (want[k][0], want[k][1], want[k][2]))
        k += 1
        _, gxs, gys = state["pyramid_last"]
        x, y, v, _ = oracle.select_from_gradients(p, gxs[0], gys[0], len(x), existing=(x, y, v))
        assert_features_equal((x, y, v), (want[k][0], want[k][1], want[k][2]))
        k += 1


def _synth(seed, shape=(480, 640), shift=(1.7, -3.3)):
    from pyfeaturetrack_b200 import synth
    return synth.frame_pair(shape[0], shape[1], seed=seed, shift=shift)


def test_synthetic_640(oracle, golden):
    imgs = _synth(0)
    p = P(oracle, max_residue=10.0, nPyramidLevels=3, subsampling=2)
    sel = oracle.select_good_features(p, imgs[0], 300)
    assert_features_equal(sel, fl(golden, "S640_sel300"))
    assert_features_equal(oracle.track_features(p, imgs[0], imgs[1], *sel)[:3], fl(golden, "S640_trk300"))
    pyr, gxs, _ = oracle.image_pyramids(p, imgs[1])
    assert np.array_equal(pyr[2], golden["S640_img1_pyr2"])
    assert np.array_equal(gxs[2], golden["S640_img1_pyr2_gradx"])


def test_synthetic_window15(oracle, golden):
    imgs = _synth(1)
    p = P(oracle, window_width=15, window_height=15, nPyramidLevels=2, subsampling=4, max_residue=8.0)
    sel = oracle.select_good_features(p, imgs[0], 200)
    assert_features_equal(sel, fl(golden, "S640w15_sel200"))
    assert_features_equal(oracle.track_features(p, imgs[0], imgs[1], *sel)[:3], fl(golden, "S640w15_trk200"))


def test_all_status_codes(oracle, golden):
    imgs = _synth(2, (240, 320), (6.2, -9.4))
    p = P(oracle, nPyramidLevels=2, subsampling=2, max_residue=5.0, max_iterations=4, min_determinant=2000.0)
    sel = oracle.select_good_features(p, imgs[0], 150)
    assert_features_equal(sel, fl(golden, "H320_sel150"))
    trk = oracle.track_features(p, imgs[0], imgs[1], *sel)[:3]
    assert_features_equal(trk, fl(golden, "H320_trk150"))
    assert set(np.unique(trk[2])) >= {0, -3, -4, -5}
    imgs = _synth(3, (240, 320))
    p = P(oracle, nPyramidLevels=2, subsampling=2, min_determinant=3.0e7)
    sel = oracle.select_good_features(p, imgs[0], 120)
    assert_features_equal(sel, fl(golden, "D320_sel120"))
    trk = oracle.track_features(p, imgs[0], imgs[1], *sel)[:3]
    assert_features_equal(trk, fl(golden, "D320_trk120"))
    assert -2 in set(np.unique(trk[2]))


def test_pairwise_sum_matches_numpy(oracle):
    """The residue uses np.abs(imgdiff).sum() in float32 (trackFeatures.py:124): pin NumPy's summation order."""
    import ctypes as C
    rng = np.random.default_rng(0)
    src = open(oracle.__file__.replace("klt_oracle.py", "klt_oracle.c")).read()
    assert "np_pairwise_sum_f32" in src
    # exercised indirectly: a window whose residue sits within an ulp of the threshold would flip the status, so
    # compare the C routine with numpy on many random vectors through a tiny shim compiled from the same source
    import subprocess, tempfile, os
    with tempfile.TemporaryDirectory() as td:
        shim = os.path.join(td, "shim.c")
        with open(shim, "w") as fh:
            fh.write('#include "%s"\nfloat shim_sum(const float*a,int n){return np_pairwise_sum_f32(a,(size_t)n);}\n'
                     % oracle.__file__.replace("klt_oracle.py", "klt_oracle.c"))
        so = os.path.join(td, "shim.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-ffp-contract=off", "-shared", "-o", so, shim, "-lm"])
        L = C.CDLL(so)
        L.shim_sum.restype = C.c_float
        L.shim_sum.argtypes = [C.POINTER(C.c_float), C.c_int]
        for n in (9, 25, 49, 81, 121, 169, 225, 441, 961):
            for _ in range(50):
                a = (rng.random(n) * 40).astype(np.float32)
                want = np.abs(a).sum()
                got = L.shim_sum(a.ctypes.data_as(C.POINTER(C.c_float)), n)
                assert np.float32(got) == want, (n, got, want)


def test_flat_image_runs_out_of_candidates(oracle):
    """Quirk Q6: the reference raises AttributeError here; like C-KLT we fill with -1 / KLT_NOT_FOUND."""
    p = P(oracle)
    img = np.full((120, 160), 77, np.uint8)
    x, y, v = oracle.select_good_features(p, img, 10)
    assert np.all(v == -1) and np.all(x == -1) and np.all(y == -1)


# ---- live comparison with the unmodified reference (only where oracle/_ref exists) ---------------------------
def test_live_reference_random_configs(oracle, reference):
    from PIL import Image
    from pyfeaturetrack_b200 import synth
    klt, sgf, tf = reference["klt"], reference["selectGoodFeatures"], reference["trackFeatures"]
    rng = np.random.default_rng(5)
    for trial in range(3):
        H, W = int(rng.integers(150, 260)), int(rng.integers(200, 330))
        imgs = synth.frame_pair(H, W, seed=10 + trial, shift=(float(rng.uniform(-3, 3)), float(rng.uniform(-3, 3))))
        kw = dict(nPyramidLevels=int(rng.integers(1, 4)), subsampling=2, max_residue=float(rng.uniform(3, 12)),
                  mindist=int(rng.integers(4, 14)), window_width=int(rng.choice([5, 7, 9])))
        kw["window_height"] = kw["window_width"]
        tc = klt.KLT_TrackingContext()
        for k, v in kw.items():
            setattr(tc, k, v)
        tc.KLTUpdateTCBorder()
        p = P(oracle, **kw)
        assert p.borderx == tc.borderx
        n = 70
        ref_fl = sgf.KLTSelectGoodFeatures(tc, Image.fromarray(imgs[0]), n)
        sel = oracle.select_good_features(p, imgs[0], n)
        assert_features_equal(sel, ([float(f.x) for f in ref_fl], [float(f.y) for f in ref_fl], [f.val for f in ref_fl]))
        tf.KLTTrackFeatures(tc, Image.fromarray(imgs[0]), Image.fromarray(imgs[1]), ref_fl)
        trk = oracle.track_features(p, imgs[0], imgs[1], *sel)[:3]
        assert_features_equal(trk, ([float(f.x) for f in ref_fl], [float(f.y) for f in ref_fl], [f.val for f in ref_fl]))


def test_oracle_equals_fullsize_goldens(oracle, golden_fullsize):
    """Config B (1080p) selection + tracking and config D's sequence with replacement against the reference's committed outputs
    (the 4K arrays are checked by the GPU suite and by test_live_reference_full_size; the scalar oracle needs ~1 min at 4K)."""
    from pyfeaturetrack_b200 import synth
    g = golden_fullsize
    imgs = synth.frame_pair(1080, 1920, seed=0)
    p = P(oracle, nPyramidLevels=3, subsampling=2, max_residue=10.0)
    sel = oracle.select_good_features(p, imgs[0], 1000)
    assert_features_equal(sel, g["B_sel1000"])
    assert_features_equal(oracle.track_features(p, imgs[0], imgs[1], *sel)[:3], g["B_trk1000"])
    nfr = 3
    shifts = [(s[0] * 6, s[1] * 6) for s in synth.sequence_shifts(5)][:nfr]
    frames = synth.frames(1080, 1920, shifts, seed=101)
    p = P(oracle, nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    x, y, v = oracle.select_good_features(p, frames[0], 1000)
    assert_features_equal((x, y, v), g["D_seq1000"][0])
    state = {}
    for k in range(1, nfr):
        x, y, v, _ = oracle.track_features(p, frames[k - 1], frames[k], x, y, v, state)
        assert_features_equal((x, y, v), g["D_seq1000"][2 * k - 1])
        _, gxs, gys = state["pyramid_last"]
        x, y, v, _ = oracle.select_from_gradients(p, gxs[0], gys[0], 1000, existing=(x, y, v))
        assert_features_equal((x, y, v), g["D_seq1000"][2 * k])


def test_live_reference_fractional_min_eigenvalue(oracle, reference):
    """tc.min_eigenvalue is compared as a number, not truncated (selectGoodFeatures.py:53,116): the reference's own
    _enforceMinimumDistance with a threshold of k + 0.5 rejects the candidates whose value is exactly k."""
    from pyfeaturetrack_b200 import synth
    klt, sgf = reference["klt"], reference["selectGoodFeatures"]
    img = synth.frames(240, 320, [(0.0, 0.0)], seed=17)[0]
    p0 = P(oracle)
    f = oracle.smooth(img.astype(np.float32), p0.smooth_sigma(), p0.cache)
    gx, gy = oracle.gradients(f, p0.grad_sigma, p0.cache)
    bx = int(p0.borderx)
    val, xs, ys = oracle.scan_good_features(gx, gy, bx, bx, 3, 3, 0)
    # integer-valued eigenvalues make the point: with cut = k + 0.5 a value of exactly k must be rejected, int(cut) = k would accept it
    val = np.floor(val).astype(np.float32)
    x, y, v, _ = oracle.select_from_gradients(p0, gx, gy, 300)
    cut = float(np.sort(v[v > 0])[150]) + 0.5
    pts = [(float(val[j, i]), int(xs[i]), int(ys[j])) for j in range(len(ys)) for i in range(len(xs))]
    pts.sort()
    pts.reverse()
    fl = []
    for _ in range(300):
        ft = klt.KLT_Feature()
        ft.x, ft.y, ft.val = -1.0, -1.0, -1
        fl.append(ft)
    sgf._enforceMinimumDistance(pts, fl, 320, 240, 10, cut, True)
    p = P(oracle, min_eigenvalue=cut)
    got = oracle.select_from_map(p, val, 320, 240, 300)
    assert_features_equal(got, ([float(t.x) for t in fl], [float(t.y) for t in fl], [t.val for t in fl]))
    assert (got[2] == -1).any() and got[2][got[2] > 0].min() > cut


@pytest.mark.parametrize("cfg", ["B", "C"])
def test_live_reference_full_size(oracle, golden, golden_fullsize, cfg):
    """The oracle against the unmodified reference at BASELINE's own sizes -- config B (1080p, 1000 features, 3 levels) selection
    + tracking and config C (4K, 10 000 features, 4 levels) selection: the float32 summed-area-table rounding grows with the
    image size (SURVEY 7.3), so this is the case that pins the selection ORDER.  Bit-identical (==).  The reference's lists
    for these inputs are stored in tests/golden/reference_golden_fullsize.npz (tests/golden/make_golden_fullsize.py)."""
    from pyfeaturetrack_b200 import synth
    H, W, n, L = (1080, 1920, 1000, 3) if cfg == "B" else (2160, 3840, 10000, 4)
    imgs = synth.frame_pair(H, W, seed=0)
    p = P(oracle, nPyramidLevels=L, subsampling=2, max_residue=10.0)
    assert [p.borderx] == [b for w, lv, ss, b in golden["borders"] if (w, lv, ss) == (7, L, 2)]
    sel = oracle.select_good_features(p, imgs[0], n)
    assert_features_equal(sel, fl(golden_fullsize, "%s_sel%d" % (cfg, n)))
    if cfg == "B":        # (tracking at 4K is covered by the GPU suite against the same stored lists)
        trk = oracle.track_features(p, imgs[0], imgs[1], *sel)[:3]
        assert_features_equal(trk, fl(golden_fullsize, "B_trk1000"))
        assert (trk[2] == 0).sum() > 900


def test_live_reference_sequence_with_replacement(oracle, reference):
    """Config D's flow against the reference itself: sequentialMode tracking + replacement through the reference's own
    _enforceMinimumDistance(..., overwriteAllFeatures=False) on tc.pyramid_last's gradients, 6 frames at 480x640."""
    from PIL import Image
    from pyfeaturetrack_b200 import synth
    klt, sgf, tf = reference["klt"], reference["selectGoodFeatures"], reference["trackFeatures"]
    nfr, n = 6, 200
    shifts = [(a * 5, b * 5) for a, b in synth.sequence_shifts(nfr)]
    frames = synth.frames(480, 640, shifts, seed=103)
    kw = dict(nPyramidLevels=3, subsampling=2, max_residue=10.0, sequentialMode=True)
    tc = klt.KLT_TrackingContext()
    for k, v in kw.items():
        setattr(tc, k, v)
    tc.KLTUpdateTCBorder()
    p = P(oracle, **kw)
    fl = sgf.KLTSelectGoodFeatures(tc, Image.fromarray(frames[0]), n)
    x, y, v = oracle.select_good_features(p, frames[0], n)
    state = {}
    replaced = 0
    for k in range(1, nfr):
        tf.KLTTrackFeatures(tc, Image.fromarray(frames[k - 1]), Image.fromarray(frames[k]), fl)
        x, y, v, _ = oracle.track_features(p, frames[k - 1], frames[k], x, y, v, state)
        assert_features_equal((x, y, v), ([float(f.x) for f in fl], [float(f.y) for f in fl], [f.val for f in fl]))
        replaced += int((v < 0).sum())
        # the reference has no public replacement entry point: drive its own pieces the way KLTReplaceLostFeatures would
        gx, gy = tc.pyramid_last_gradx.img[0], tc.pyramid_last_grady.img[0]
        bx = int(max(tc.borderx, tc.window_width / 2)); hw = int(tc.window_width / 2)
        import goodFeaturesUtils as rgfu
        px, py, pv = rgfu.ScanImageForGoodFeatures(gx, gy, bx, bx, hw, hw, tc.nSkippedPixels)
        pts = list(zip(pv, px, py)); pts.sort(); pts.reverse()
        sgf._enforceMinimumDistance(pts, fl, 640, 480, tc.mindist, tc.min_eigenvalue, False)
        _, gxs, gys = state["pyramid_last"]
        x, y, v, _ = oracle.select_from_gradients(p, gxs[0], gys[0], n, existing=(x, y, v))
        assert_features_equal((x, y, v), ([float(f.x) for f in fl], [float(f.y) for f in fl], [f.val for f in fl]))
    assert replaced > 0


# ---- affine consistency check: unpinned by the reference (its callees are undefined there); property tests only -------
def _affine_sequence(n_frames=5, H=360, W=480):
    """Frames of one texture under a growing rotation + scale + shift (known ground truth)."""
    import scipy.ndimage as ndi
    from pyfeaturetrack_b200 import synth
    base = synth._texture(H, W, 7)
    c = np.array([64 + H / 2, 64 + W / 2])
    raw = []
    for k in range(n_frames):
        a, s = 0.01 * k, 1 + 0.004 * k
        M = s * np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
        off = c - M @ c + np.array([0.6 * k, -0.9 * k])
        raw.append(ndi.affine_transform(base, M, offset=off, order=3, mode="reflect")[64:-64, 64:-64])
    lo, hi = raw[0].min(), raw[0].max()
    return [np.clip((f - lo) * 255 / (hi - lo), 0, 255).astype(np.uint8) for f in raw]


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_affine_restatement_recovers_known_warp(oracle, mode):
    frames = _affine_sequence()
    p = P(oracle, nPyramidLevels=2, subsampling=2, max_residue=10.0, affineConsistencyCheck=mode)
    p.borderx = p.bordery = max(p.borderx, 12.0)
    x, y, v = oracle.select_good_features(p, frames[0], 120)
    aff = oracle.AffineState(120)
    for k in range(1, len(frames)):
        x, y, v, _ = oracle.track_features_affine(p, frames[k - 1], frames[k], x, y, v, aff)
        if k == 1:
            assert aff.has.sum() == (v == 0).sum() and np.all(aff.A == (1, 0, 0, 1))     # first track only stores templates
            live = v == 0
            assert np.all((aff.aff_x[live] >= 8) & (aff.aff_x[live] < 9))                  # frac + (15+2)//2
    live = v == 0
    assert live.mean() > 0.9
    a, s = 0.01 * 4, 1 + 0.004 * 4
    want = np.array([np.cos(a) / s, np.sin(a) / s, -np.sin(a) / s, np.cos(a) / s])       # inverse of the resampling map
    got = aff.A[live].mean(0)
    if mode == 0:
        assert np.all(aff.A[live] == (1, 0, 0, 1))
    else:
        assert np.abs(got - want).max() < 5e-3, (got, want)
    # lost features have no template and aff_x = aff_y = -1 once the affine tracker rejected them
    assert np.all(aff.has[~live] == 0)
