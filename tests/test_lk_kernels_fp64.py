"""The FAST and windowed Lucas-Kanade trackers against a float64 reference, one Newton step at a time.

With retain_trackers = 1, min_displacement = 0 and max_iterations = k, a one-level track runs exactly k Newton steps and
returns the position after step k (only the final border check can still clear it).  The kernels are deterministic, so
tracks with k = 1 .. K return the GPU's own iterates x_1 .. x_K.  Each GPU step x_k -> x_k+1 is compared with one float64
step taken from the GPU's own x_k, so errors do not compound and no convergence analysis is needed.

The reference step (per feature, vectorised): bilinear samples with the exact weights of ax = x - floor(x);
diff = T - P, g = Tg + Pg, G = sum [gx^2, gx gy; gx gy, gy^2], e = step_factor * sum diff [gx, gy], d = G^-1 e (the sign
conventions of iterate_exact in klt_track.cu).  Inputs are the GPU's own planes: for FAST pyramids the intensity and
gradient planes exactly; for image-only (windowed) pyramids the intensity plane exactly and the gradients the kernel
evaluates in its windows, emulated in float32 in its operation order (windowed_gradients), with a margin of 2u |g|.

Error bound: running error analysis in the standard model (|delta| <= u |result| per rounding, u = 2**-24), an absolute
bound carried along every quantity and evaluated in float64 per feature:
  * bilinear sample: the weight errors plus the 4-term FMA chain (4u max|p|) plus the input error.  The kernels form
    w11 = ax ay, w01 = ax - w11, w10 = ay - w11 and w00 = ((1 - ax) - ay) + w11 from the exact ax, ay: w11's rounding
    reaches all four weights, each also rounds once and w00 twice more on values <= 1, so
    sum |dw| <= u (4 w11 + w01 + w10 + w00 + 2) <= 6u, and the sample is off by at most 10u max|p|.  The exact-order
    kernel's bilerp_ref (double products, one float product, one rounding to float): 4u max|p|;
  * diff and g: the operand errors plus one rounding;
  * the five sums: sum of first-order product errors + gamma_m sum |terms|, m the rounding depth of the kernel's reduction
    (lk_track_rows: W FMAs per lane + log2 G shuffle levels; lk_windowed: PX FMAs + log2 LPF levels; lk_track: n sequential
    adds + the product);
  * det and the numerators: first-order propagation plus their roundings;
  * dx: (e_num + |dx| e_det) / (|det| - e_det) + 2u |dx| (a division, or a reciprocal and a product);
  * position: u |x_new|.
Contraction into FMA by the compiler only removes roundings, so the bound holds whether or not it happens.  Features with
det <= 2 e_det are ill-conditioned: they are dropped from the position checks and counted.

Every GPU case asserts through the launch profile which tracker ran.  Run with -s to see each check's largest err / bound
and the median position bound."""
import ctypes as C
import math

import numpy as np
import pytest

from test_fast_kernels_fp64 import (U, conv_separable, gradients, make_tc, pass_bound, profiled, random_frames, reflect_index,
                                    taps_for)

TRACKED, SMALL_DET, MAX_ITERATIONS, OOB, LARGE_RESIDUE = 0, -2, -3, -4, -5
f32 = np.float32
K_STEPS = 5
RATIOS = {}
POS_BOUNDS = {}


def record(kind, err, bound, label):
    """err <= bound elementwise; prints and records the largest ratio per kind."""
    err, bound = np.asarray(err, np.float64), np.asarray(bound, np.float64)
    ratio = float((err / bound).max()) if err.size else 0.0
    RATIOS[kind] = max(RATIOS.get(kind, 0.0), ratio)
    if err.size:
        print("fp64 %-64s n %5d  max err %.3e  median bound %.3e  err/bound %.3f" % (label, err.size, err.max(),
                                                                                      np.median(bound), ratio))
    bad = err > bound
    assert not bad.any(), "%s: %d of %d above their bound (largest ratio %.3f)" % (label, bad.sum(), err.size, ratio)


@pytest.fixture(scope="module", autouse=True)
def _ratio_summary():
    yield
    if RATIOS:
        print("\nfp64 largest err/bound per kernel and check: " + ", ".join("%s %.3f" % kv for kv in sorted(RATIOS.items())))
    for k, v in sorted(POS_BOUNDS.items()):
        print("fp64 median position bound %s: %.3e px over %d steps" % (k, np.median(np.concatenate(v)), sum(map(len, v))))


# ---- the float64 reference step and its bound ------------------------------------------------------------------------------
def depth(kind, W):
    """Rounding depth of the kernel's window sums (module docstring)."""
    if kind == "lk_track_rows":
        return W + int(math.log2(8 if W <= 7 else 16))
    if kind == "lk_windowed":
        lpf = 32 // (2 if W <= 7 else 1)
        rpr = lpf // (4 if W <= 4 else (8 if W <= 8 else 16))
        return -(-W // rpr) + int(math.log2(lpf))
    return W * W + 1


class Level:
    """float64 inputs of one pyramid level, (B, H, W) per plane.  e1 / e2: input error of the gradient planes, one number
    per image or per pixel as a pair of (B, H, W) planes (gx, gy)."""

    def __init__(self, I1, GX1, GY1, e1, I2, GX2, GY2, e2):
        def planes(e, I):
            if isinstance(e, tuple):
                return e
            e = np.broadcast_to(np.asarray(e, np.float64)[:, None, None], I.shape)
            return e, e
        self.I1, self.GX1, self.GY1, self.I2, self.GX2, self.GY2 = I1, GX1, GY1, I2, GX2, GY2
        (self.EX1, self.EY1), (self.EX2, self.EY2) = planes(e1, I1), planes(e2, I2)


def sample(P, img, x, y, W):
    """Bilinear W x W window of planes P[img] at (x, y) with the exact weights; also max|tap| of each sample's footprint."""
    x, y = np.asarray(x, np.float64), np.asarray(y, np.float64)
    ix, iy = np.floor(x).astype(np.int64), np.floor(y).astype(np.int64)
    ax, ay = (x - ix)[:, None, None], (y - iy)[:, None, None]
    o = np.arange(W) - W // 2
    R, Cc, I = (iy[:, None] + o)[:, :, None], (ix[:, None] + o)[:, None, :], np.asarray(img)[:, None, None]
    a, b, c, d = P[I, R, Cc], P[I, R, Cc + 1], P[I, R + 1, Cc], P[I, R + 1, Cc + 1]
    v = (1 - ax) * (1 - ay) * a + ax * (1 - ay) * b + (1 - ax) * ay * c + ax * ay * d
    M = np.maximum(np.maximum(np.abs(a), np.abs(b)), np.maximum(np.abs(c), np.abs(d)))
    return v, M


def prod_err(a, ea, b, eb):
    return np.abs(a) * eb + np.abs(b) * ea + ea * eb


class Step:
    """One float64 Newton step from (x2, y2) with the template at (x1, y1), with the bounds of `kind`'s fp32 arithmetic."""

    def __init__(self, lv, img, x1, y1, x2, y2, W, kind, step_factor=1.0):
        cs = 4.01 * U if kind == "lk_track" else 10.01 * U
        img = np.asarray(img)
        T, MT = sample(lv.I1, img, x1, y1, W)
        Tx, MTx = sample(lv.GX1, img, x1, y1, W)
        Ty, MTy = sample(lv.GY1, img, x1, y1, W)
        P, MP = sample(lv.I2, img, x2, y2, W)
        Px, MPx = sample(lv.GX2, img, x2, y2, W)
        Py, MPy = sample(lv.GY2, img, x2, y2, W)
        # input errors of the gradient samples: the largest of the four taps' (the weights sum to 1)
        (_, eX1), (_, eY1) = sample(lv.EX1, img, x1, y1, W), sample(lv.EY1, img, x1, y1, W)
        (_, eX2), (_, eY2) = sample(lv.EX2, img, x2, y2, W), sample(lv.EY2, img, x2, y2, W)
        eT, eTx, eTy = cs * MT, cs * MTx + eX1, cs * MTy + eY1
        eP, ePx, ePy = cs * MP, cs * MPx + eX2, cs * MPy + eY2
        diff, gx, gy = T - P, Tx + Px, Ty + Py
        ed = eT + eP + U * (np.abs(diff) + eT + eP)
        egx = eTx + ePx + U * (np.abs(gx) + eTx + ePx)
        egy = eTy + ePy + U * (np.abs(gy) + eTy + ePy)
        m = depth(kind, W)
        gam = m * U / (1 - m * U)

        def wsum(a, ea, b, eb):
            s = (a * b).sum((1, 2))
            e = prod_err(a, ea, b, eb).sum((1, 2)) + gam * ((np.abs(a) + ea) * (np.abs(b) + eb)).sum((1, 2))
            return s, e
        gxx, Exx = wsum(gx, egx, gx, egx)
        gxy, Exy = wsum(gx, egx, gy, egy)
        gyy, Eyy = wsum(gy, egy, gy, egy)
        ex, Eex = wsum(diff, ed, gx, egx)
        ey, Eey = wsum(diff, ed, gy, egy)
        sf = abs(float(step_factor))
        ex, ey = ex * step_factor, ey * step_factor
        Eex, Eey = sf * Eex + U * (np.abs(ex) + sf * Eex), sf * Eey + U * (np.abs(ey) + sf * Eey)

        def cross(a, ea, b, eb, c, ec, d, ed_):      # a b - c d with its error: the operands', two products, one difference
            mag = (np.abs(a) + ea) * (np.abs(b) + eb) + (np.abs(c) + ec) * (np.abs(d) + ed_)
            return a * b - c * d, prod_err(a, ea, b, eb) + prod_err(c, ec, d, ed_) + 2.01 * U * mag
        self.det, self.e_det = cross(gxx, Exx, gyy, Eyy, gxy, Exy, gxy, Exy)
        nx, e_nx = cross(gyy, Eyy, ex, Eex, gxy, Exy, ey, Eey)
        ny, e_ny = cross(gxx, Exx, ey, Eey, gxy, Exy, ex, Eex)
        self.ok = self.det > 2 * self.e_det                                  # well-conditioned
        den = np.where(self.ok, self.det - self.e_det, np.inf)
        det = np.where(self.det != 0, self.det, 1.0)
        self.dx, self.dy = nx / det, ny / det
        bx = (e_nx + np.abs(self.dx) * self.e_det) / den
        by = (e_ny + np.abs(self.dy) * self.e_det) / den
        bx, by = bx + 2.01 * U * (np.abs(self.dx) + bx), by + 2.01 * U * (np.abs(self.dy) + by)
        self.e_dx, self.e_dy = bx, by
        self.x = np.asarray(x2, np.float64) + self.dx
        self.y = np.asarray(y2, np.float64) + self.dy
        self.e_x = bx + 1.01 * U * (np.abs(self.x) + bx)
        self.e_y = by + 1.01 * U * (np.abs(self.y) + by)
        # residue mean|T - P| at (x2, y2): the per-pixel errors, one rounding per difference, the sum's depth, the division
        n = W * W
        ad = np.abs(diff)
        self.res = ad.sum((1, 2)) / n
        s = (ad + eT + eP).sum((1, 2)) / n
        self.e_res = (eT + eP).sum((1, 2)) / n + (U + gam) * s + 1.01 * U * s


# ---- what the kernels decide, restated exactly (float32 / float64 as the kernels compute it) ---------------------------------
def loop_oob(x, y, W, nc, nr):
    """The in-loop check of every tracker: float32, integer hw."""
    x, y, hw = f32(x), f32(y), f32(W // 2)
    with np.errstate(over="ignore"):
        return (x - hw < 0) | (f32(nc) - (x + hw) < f32(1.001)) | (y - hw < 0) | (f32(nr) - (y + hw) < f32(1.001))


def post_oob(x, y, W, nc, nr):
    """The post-loop check in doubles with hw = W / 2.0 (quirk Q2)."""
    x, y, hw = np.float64(f32(x)), np.float64(f32(y)), W / 2.0
    return (x - hw < 0) | (nc - (x + hw) < 1.001) | (y - hw < 0) | (nr - (y + hw) < 1.001)


def border_oob(x, y, W0, H0, bx, by):
    return (x < bx) | (x > (W0 - 1) - bx) | (y < by) | (y > (H0 - 1) - by)


def template_assert(x, y, W, nc, nr):
    ix, iy, hw = np.trunc(f32(x)).astype(np.int64), np.trunc(f32(y)).astype(np.int64), W // 2
    return ~((ix - hw >= 0) & (iy - hw >= 0) & (ix + hw + 2 <= nc) & (iy + hw + 2 <= nr))


# ---- CPU: the reference step against the oracle, and the bound against float32 emulations ------------------------------------
def smooth_pair(seed, H, W, shift, rough=False):
    """Float planes of a frame pair: intensity (the FAST level-0 smoothing) and its gradients, as float32.  rough: random
    u8 texture, shifted with cubic interpolation (gradients of tens of units per pixel instead of a few)."""
    import scipy.ndimage as ndi
    from pyfeaturetrack_b200 import synth
    _, T = taps_for(nPyramidLevels=1, subsampling=2)
    if rough:
        f = random_frames(seed, 1, H, W)[0].astype(np.float64)
        pair = (f, ndi.shift(f, shift, order=3, mode="reflect"))
    else:
        pair = synth.frame_pair(H, W, seed=seed, shift=shift)
    out = []
    for f in pair:
        I = conv_separable(f.astype(np.float64), T.s, T.s)
        gx, gy = gradients(I, T.g, T.d)
        out.append((I.astype(f32), gx.astype(f32), gy.astype(f32)))
    return out


def interior_starts(rng, n, W, nc, nr, margin):
    hw = W // 2
    x = rng.uniform(hw + margin, nc - hw - 1.001 - margin, n).astype(f32)
    y = rng.uniform(hw + margin, nr - hw - 1.001 - margin, n).astype(f32)
    return x.astype(np.float64), y.astype(np.float64)


@pytest.mark.parametrize("W", [3, 7, 15, 17])
def test_reference_step_matches_oracle(oracle, W):
    """oracle.track_on_pyramids (bit-exact with the original) with retainTrackers, min_displacement 0 and max_iterations
    1, 2, 3 on float planes: each of its steps is within the exact-order bound of the reference step taken from its own
    previous iterate.  The steps are far larger than the bound, so a sign or orientation slip cannot hide in it."""
    H, Wd = 64, 88
    (I1, X1, Y1), (I2, X2, Y2) = smooth_pair(W, H, Wd, (0.9, -1.3))
    lv = Level(*(a[None].astype(np.float64) for a in (I1, X1, Y1)), [0.0], *(a[None].astype(np.float64) for a in (I2, X2, Y2)), [0.0])
    rng = np.random.default_rng(W)
    n = 60
    x0, y0 = interior_starts(rng, n, W, Wd, H, 4)
    p = oracle.Params(window_width=W, window_height=W, nPyramidLevels=1, retainTrackers=True, min_displacement=0.0)
    p.borderx = p.bordery = 0.0
    pyr1, pyr2 = ([I1], [X1], [Y1]), ([I2], [X2], [Y2])
    prev = (x0, y0, np.zeros(n, np.int32))
    img = np.zeros(n, np.int64)
    checked = 0
    for k in (1, 2, 3):
        p.max_iterations = k
        x, y, v, _ = oracle.track_on_pyramids(p, pyr1, pyr2, x0, y0, np.zeros(n, np.int32))
        live = (prev[2] == 0) & ~loop_oob(prev[0], prev[1], W, Wd, H)
        s = Step(lv, img[live], x0[live], y0[live], prev[0][live], prev[1][live], W, "lk_track")
        good = s.ok & (s.det - s.e_det >= p.min_determinant) & (v[live] == 0)
        assert good.mean() > 0.9
        record("lk_track oracle", np.abs(x[live][good] - s.x[good]), s.e_x[good], "oracle W%d step %d x" % (W, k))
        record("lk_track oracle", np.abs(y[live][good] - s.y[good]), s.e_y[good], "oracle W%d step %d y" % (W, k))
        assert np.median(np.abs(s.dx[good]) + np.abs(s.dy[good])) > 1e3 * np.median(s.e_x[good])
        checked += good.sum()
        prev = (x, y, v)
    assert checked > 150


def emulate_rows_step(I1, X1, Y1, I2, X2, Y2, x1, y1, x2, y2, W, mutation=None):
    """One Newton step of lk_track_rows in float32, in the kernel's operation order (one image; planes float32)."""
    def fma(a, b, c):
        return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(f32)

    def weights(x, y):
        ix, iy = np.floor(x).astype(np.int64), np.floor(y).astype(np.int64)
        ax, ay = f32(x) - ix.astype(f32), f32(y) - iy.astype(f32)
        w11 = ax * ay
        w00 = (f32(1) - ax - ay) if mutation == "w00 without w11" else (f32(1) - ax - ay + w11)
        return ix, iy, [a[:, None, None] for a in (w00, ax - w11, ay - w11, w11)]

    def patch(Pl, ix, iy, w):
        o = np.arange(W) - W // 2
        R, Cc = (iy[:, None] + o)[:, :, None], (ix[:, None] + o)[:, None, :]
        a, b, c, d = Pl[R, Cc], Pl[R, Cc + 1], Pl[R + 1, Cc], Pl[R + 1, Cc + 1]
        w00, w01, w10, w11 = w
        return fma(w11, d, fma(w10, c, fma(w01, b, w00 * a)))

    i1 = weights(x1, y1)
    i2 = weights(x2, y2)
    if mutation == "tap scaled":
        i2[2][0] = i2[2][0] * f32(1 + 1e-5)
    T, Tx, Ty = patch(I1, i1[0], i1[1], i1[2]), patch(X1, i1[0], i1[1], i1[2]), patch(Y1, i1[0], i1[1], i1[2])
    P, Px, Py = patch(I2, i2[0], i2[1], i2[2]), patch(X2, i2[0], i2[1], i2[2]), patch(Y2, i2[0], i2[1], i2[2])
    diff, gx, gy = T - P, Tx + Px, Ty + Py
    rows = W - 1 if mutation == "row dropped" else W
    G = 8 if W <= 7 else 16
    sums = []
    for a, b in ((gx, gx), (gx, gy), (gy, gy), (diff, gx), (diff, gy)):
        lane = np.zeros((a.shape[0], G), f32)                 # lane j: column j, the rows in order
        for i in range(rows):
            lane[:, :W] = fma(a[:, i, :], b[:, i, :], lane[:, :W])
        o = 1
        while o < G:                                          # the xor butterfly of group_sum<G>
            lane = lane + lane[:, np.arange(G) ^ o]
            o <<= 1
        sums.append(lane[:, 0])
    gxx, gxy, gyy, ex, ey = sums
    det = gxx * gyy - gxy * gxy
    dx = (gyy * ex - gxy * ey) / det
    dy = (gxx * ey - gxy * ex) / det
    return f32(x2) + dx, f32(y2) + dy


@pytest.mark.parametrize("W", [3, 7, 9, 15])
def test_bound_admits_rows_emulation_and_rejects_mutants(W):
    """A float32 emulation of one lk_track_rows step meets the bound; emulations with the w00 tap of the second image's
    bilinear samples scaled by 1 + 1e-5 (up to 9 x 9: at 15 x 15 the bound allows for 225 sample errors adding up and
    the scaled tap stays inside it), one window row dropped, or w11 left out of w00 do not."""
    H, Wd = 72, 96
    (I1, X1, Y1), (I2, X2, Y2) = smooth_pair(40 + W, H, Wd, (1.1, 0.7), rough=True)
    lv = Level(*(a[None].astype(np.float64) for a in (I1, X1, Y1)), [0.0], *(a[None].astype(np.float64) for a in (I2, X2, Y2)), [0.0])
    rng = np.random.default_rng(W)
    n = 300
    x1, y1 = interior_starts(rng, n, W, Wd, H, 4)
    x2 = (x1 + rng.uniform(-3, 3, n)).astype(f32).astype(np.float64)
    y2 = (y1 + rng.uniform(-3, 3, n)).astype(f32).astype(np.float64)
    s = Step(lv, np.zeros(n, np.int64), x1, y1, x2, y2, W, "lk_track_rows")
    ok = s.ok
    assert ok.mean() > 0.95

    def ratio(mutation):
        gx_, gy_ = emulate_rows_step(I1, X1, Y1, I2, X2, Y2, x1, y1, x2, y2, W, mutation)
        return max(float((np.abs(gx_[ok] - s.x[ok]) / s.e_x[ok]).max()), float((np.abs(gy_[ok] - s.y[ok]) / s.e_y[ok]).max()))
    r = ratio(None)
    print("fp64 rows emulation W%d: err/bound %.3f" % (W, r))
    assert r <= 1.0
    for mutation in (("tap scaled",) if W <= 9 else ()) + ("row dropped", "w00 without w11"):
        rm = ratio(mutation)
        print("fp64 rows emulation W%d, %s: err/bound %.3f" % (W, mutation, rm))
        assert rm > 1.0, mutation


def test_windowed_gradient_emulation():
    """windowed_gradients: fmaf rounds correctly (against exact rationals), and the emulated planes lie within the fp32
    pass bound of the float64 gradients, for unequal gradient taps too."""
    from fractions import Fraction
    rng = np.random.default_rng(1)
    a, b, c = (rng.standard_normal(3000).astype(f32) for _ in range(3))
    c[:1000] = -(a[:1000] * b[:1000])                   # heavy cancellation
    got = fmaf(a, b, c)
    for i in range(0, 3000, 7):
        x = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        near = [f32(float(x))]
        near += [np.nextafter(near[0], f32(np.inf)), np.nextafter(near[0], f32(-np.inf))]
        best = min(near, key=lambda v: (abs(Fraction(float(v)) - x), int(np.asarray(v).view(np.uint32)) & 1))
        assert got[i] == best, i
    for sigma in (1.0, 1.1):
        _, T = taps_for(nPyramidLevels=1, subsampling=2, grad_sigma=sigma)
        I = random_frames(3, 1, 37, 53)[0].astype(np.float64)
        gx, gy = windowed_gradients(I, T)
        wx, wy = gradients(I, T.g, T.d)
        b = pass_bound(T.d, T.g, 0.0, 255.0)
        assert np.abs(gx - wx).max() <= b and np.abs(gy - wy).max() <= b
        assert np.abs(gx - wx).max() > 0                # it does round


# ---- GPU cases --------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


def track(ctx, params, p1, p2, n_per_image, x, y, v):
    """klt_track_features on copies of the lists; returns (x, y, val, n_iterations)."""
    from pyfeaturetrack_b200 import _capi
    x, y, v = np.array(x, np.float64), np.array(y, np.float64), np.array(v, np.int32)
    it = C.c_int64()
    ctx.check(_capi.lib().klt_track_features(ctx.handle, C.byref(params), p1.handle, p2.handle, n_per_image, x.ctypes.data,
                                             y.ctypes.data, v.ctypes.data, C.byref(it)))
    return x, y, v, it.value


def tracker_of(ran):
    return {k for k in ran if k.startswith("lk_")}


def make_params(W, L=1, ss=2, **kw):
    from pyfeaturetrack_b200 import selectGoodFeatures as sgf
    p = sgf.make_params(make_tc(window_width=W, window_height=W, nPyramidLevels=L, subsampling=ss))
    p.borderx = p.bordery = 0.0
    p.has_max_residue = 0
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def fmaf(a, b, c):
    """Correctly rounded float32 fma(a, b, c), elementwise: a b is exact in float64, TwoSum gives the error of the float64
    sum, and only a sum that lands exactly on a float32 rounding midpoint needs that error to pick its side."""
    p = np.asarray(a, np.float64) * np.asarray(b, np.float64)
    c = np.asarray(c, np.float64)
    s = p + c
    bb = s - p
    e = (p - (s - bb)) + (c - bb)
    r = s.astype(f32)
    r64 = r.astype(np.float64)
    up, dn = np.nextafter(r, f32(np.inf)), np.nextafter(r, f32(-np.inf))
    r = np.where((s == (r64 + up.astype(np.float64)) / 2) & (e > 0), up, r)
    return np.where((s == (r64 + dn.astype(np.float64)) / 2) & (e < 0), dn, r)


def windowed_gradients(I, T):
    """gx, gy of a level as lk_windowed evaluates them in its windows, emulated in float32 in the kernel's operation order
    (gradient_pair): the float taps flip7 hands it (K.g[k] multiplies in[x + k - 3]); the vertical pass first (Gaussian
    for gx, derivative for gy) as a product and six FMAs per output, then the horizontal one the same way; 'reflect'
    borders.  Every output depends only on its pixel, not on the window that computed it.  A float64 reference would
    have to allow each value the pass's rounding, about 1e-4 at intensities near 128: more than a tap that is 1e-5 off
    changes a gradient of these frames by, so the gradient-tap mutations would pass unseen."""
    H, W = I.shape
    g, d = np.asarray(T.g[::-1], f32), np.asarray(T.d[::-1], f32)
    Ir = np.asarray(I, f32)[reflect_index(np.arange(-3, H + 3), H)][:, reflect_index(np.arange(-3, W + 3), W)]

    def vpass(k):
        t = k[0] * Ir[0:H]
        for j in range(1, 7):
            t = fmaf(k[j], Ir[j:j + H], t)
        return t

    def hpass(t, k):
        acc = k[0] * t[:, 0:W]
        for j in range(1, 7):
            acc = fmaf(k[j], t[:, j:j + W], acc)
        return acc
    return hpass(vpass(g), d).astype(np.float64), hpass(vpass(d), g).astype(np.float64)


def level_inputs(p1, p2, T1, T2, B, windowed, lvl=0):
    """The reference's inputs at one level: the GPU's own planes.  Call only after the last track on these pyramids: a
    gradient download builds the planes of an image-only pyramid and sends every later track to lk_track_rows."""
    out = []
    for pyr, T in ((p1, T1), (p2, T2)):
        I = np.stack([pyr.download(0, lvl, b) for b in range(B)]).astype(np.float64)
        if windowed:
            g = [windowed_gradients(I[b], T) for b in range(B)]
            GX, GY = np.stack([a for a, _ in g]), np.stack([b for _, b in g])
            e = (2 * U * np.abs(GX), 2 * U * np.abs(GY))     # a margin of 2u: the emulation is meant to be exact
        else:
            GX = np.stack([pyr.download(1, lvl, b) for b in range(B)]).astype(np.float64)
            GY = np.stack([pyr.download(2, lvl, b) for b in range(B)]).astype(np.float64)
            e = np.zeros(B)
        out += [I, GX, GY, e]
    return Level(*out)


def start_positions(seed, B, n, W, nc, nr):
    """Per image: every 8th feature dead (val -1), the others in the interior or within hw + 3 px of one of the four edges
    (the windowed kernel then stages both images by its 'reflect' element path), as float32 values."""
    rng = np.random.default_rng(seed)
    hw = W // 2
    N = B * n
    x, y = interior_starts(rng, N, W, nc, nr, 8)
    kind = np.arange(N) % 8
    lo, hi_x, hi_y = hw + rng.uniform(0, 3, N), nc - hw - 1.001 - rng.uniform(0, 3, N), nr - hw - 1.001 - rng.uniform(0, 3, N)
    x = np.where(kind == 1, lo, np.where(kind == 2, hi_x, x))
    y = np.where(kind == 3, lo, np.where(kind == 4, hi_y, y))
    x, y = x.astype(f32).astype(np.float64), y.astype(f32).astype(np.float64)
    v = np.where(kind == 7, -1, 0).astype(np.int32)
    v[np.arange(N) % n == 0] = 0                 # the first feature of every image is alive
    return x, y, v


def expected_tracker(W, windowed):
    if windowed:
        return "lk_windowed"
    return "lk_track_rows" if W <= 15 else "lk_track"


def run_iterates(ctx, params, p1, p2, n_per_image, x0, y0, v0, K, want):
    """Tracks with max_iterations = 1 .. K (and K again: bit-identical); returns [(x, y, val, n_iterations)] for k = 0 .. K."""
    out = [(x0, y0, v0, 0)]
    for k in range(1, K + 1):
        params.max_iterations = k
        ran = profiled(ctx, lambda: out.append(track(ctx, params, p1, p2, n_per_image, x0, y0, v0)))
        assert tracker_of(ran) == {want}, (sorted(ran), want)
    again = track(ctx, params, p1, p2, n_per_image, x0, y0, v0)
    assert all(np.array_equal(a, b) for a, b in zip(again[:3], out[-1][:3])) and again[3] == out[-1][3]
    dead = v0 < 0
    for x, y, v, _ in out:
        assert np.array_equal(x[dead], x0[dead]) and np.array_equal(y[dead], y0[dead]) and np.array_equal(v[dead], v0[dead])
    return out


def check_iterates(lv, iters, W, kind, n_per_image, nc, nr, small_det, label, step_factor=1.0):
    """Every GPU step x_k -> x_k+1 against the reference step from the GPU's own x_k; the iteration counts of the tracks."""
    x0, y0, v0, _ = iters[0]
    N = len(x0)
    img = np.arange(N) // n_per_image
    running_lo, running_hi = v0 >= 0, v0 >= 0          # surely / possibly still iterating in the track with max_iterations = k
    it_lo = it_hi = 0
    n_ill = n_steps = n_exact = 0
    for k in range(1, len(iters)):
        (px, py, pv, _), (x, y, v, its) = iters[k - 1], iters[k]
        lost = (pv == OOB) & (v0 >= 0)
        assert (v[lost] == OOB).all(), label                      # once outside the image, the track stops there
        live = pv == TRACKED
        oob = live & loop_oob(px, py, W, nc, nr)
        assert (v[oob] == TRACKED).all() and np.array_equal(x[oob], px[oob]) and np.array_equal(y[oob], py[oob]), label
        st = live & ~oob
        idx = np.nonzero(st)[0]
        s = Step(lv, img[idx], x0[idx], y0[idx], px[idx], py[idx], W, kind, step_factor)
        ill = ~s.ok
        still = s.ok & (s.det + s.e_det < small_det)
        took = s.ok & (s.det - s.e_det >= small_det)
        n_ill += ill.sum()
        f_still = idx[still]
        assert np.array_equal(x[f_still], px[f_still]) and np.array_equal(y[f_still], py[f_still]), label
        on = took & (v[idx] == TRACKED)
        record(kind + " step", np.abs(x[idx][on] - s.x[on]), s.e_x[on], "%s k%d x" % (label, k))
        record(kind + " step", np.abs(y[idx][on] - s.y[on]), s.e_y[on], "%s k%d y" % (label, k))
        POS_BOUNDS.setdefault(kind, []).append(np.concatenate([s.e_x[on], s.e_y[on]]))
        n_steps += on.sum()
        gone = took & (v[idx] == OOB)               # the step left the image: the final border check (0 here) cleared it
        if gone.any():
            could = border_oob(s.x[gone] - s.e_x[gone], s.y[gone] - s.e_y[gone], nc, nr, 0, 0) | \
                border_oob(s.x[gone] + s.e_x[gone], s.y[gone] + s.e_y[gone], nc, nr, 0, 0)
            assert could.all(), label
        assert np.isin(v[idx][took], (TRACKED, OOB)).all(), label
        sure = np.zeros(N, bool)
        maybe = np.zeros(N, bool)
        sure[idx[took]] = True
        maybe[idx[took | ill | ~(still | took)]] = True
        running_lo = running_lo & sure
        running_hi = running_hi & (sure | maybe)
        it_lo += running_lo.sum()
        it_hi += running_hi.sum()
        if it_lo == it_hi:             # every decision outside its bound: the count is known exactly
            assert its == it_lo, (label, k, its, it_lo)
            n_exact += 1
        assert it_lo <= its <= it_hi, (label, k, it_lo, its, it_hi)
    alive = (v0 >= 0).sum()
    print("fp64 %s: %d steps checked, %d ill-conditioned of %d features x %d steps, iteration count exact in %d of %d tracks"
          % (label, n_steps, n_ill, alive, len(iters) - 1, n_exact, len(iters) - 1))
    assert n_ill <= 0.05 * alive * (len(iters) - 1), label
    assert n_steps >= 0.2 * alive * (len(iters) - 1), label


MOTIONS = {"0.6px": (0.4, 0.6), "2.5px": (-1.5, 2.5), "4.5px": (2.0, -4.5), "random": None}


def frames_for(motion, B, H, W, seed):
    from pyfeaturetrack_b200 import synth
    if MOTIONS[motion] is None:
        return random_frames(seed, B, H, W), random_frames(seed + 1, B, H, W)
    f1, f2 = np.empty((B, H, W), np.uint8), np.empty((B, H, W), np.uint8)
    for b in range(B):
        f1[b], f2[b] = synth.frame_pair(H, W, seed=seed + b, shift=MOTIONS[motion])
    return f1, f2


def step_case(ctx, f1, f2, W, windowed, label, n_per_image=37, taps2=None, seed=0, f32_input=False):
    """Builds the pair (u8 frames, or float images as already-smoothed level 0), tracks K_STEPS iterates and checks them."""
    from pyfeaturetrack_b200 import _capi
    B, H, Wd = f1.shape
    t1, T1 = taps_for(nPyramidLevels=1, subsampling=2, window_width=W, window_height=W)
    t2, T2 = taps2 if taps2 is not None else (t1, T1)
    prec = _capi.PRECISION_FAST_WINDOWED if windowed else _capi.PRECISION_FAST
    p1, p2 = _capi.Pyramid(ctx, Wd, H, 1, 2, B), _capi.Pyramid(ctx, Wd, H, 1, 2, B)
    try:
        for pyr, f, t in ((p1, f1, t1), (p2, f2, t2)):
            if f32_input:
                ran = profiled(ctx, lambda: pyr.build_f32(f, t, prec, 1))
                assert not windowed or not any("grad" in k for k in ran), sorted(ran)   # image-only: no gradient plane
            else:
                pyr.build_u8(f, t, prec)
        params = make_params(W, retain_trackers=1, min_displacement=0.0)
        x0, y0, v0 = start_positions(seed, B, n_per_image, W, Wd, H)
        iters = run_iterates(ctx, params, p1, p2, n_per_image, x0, y0, v0, K_STEPS, expected_tracker(W, windowed))
        lv = level_inputs(p1, p2, T1, T2, B, windowed)
    finally:
        p1.close(); p2.close()
    kind = expected_tracker(W, windowed)
    check_iterates(lv, iters, W, kind, n_per_image, Wd, H, params.min_determinant, label)
    return lv, iters


@gpu
@pytest.mark.parametrize("motion", list(MOTIONS))
@pytest.mark.parametrize("W,windowed", [(w, False) for w in (3, 5, 7, 9, 11, 13, 15, 17, 21)] +
                         [(w, True) for w in (3, 5, 7, 9, 11, 13, 15)])
def test_newton_steps(gpu_ctx, W, windowed, motion):
    """lk_track_rows (W <= 15) and lk_track (17, 21) on FAST pyramids, lk_windowed on image-only ones: a batch of 3 images
    of 157 x 203 (widths not a multiple of 4) with 37 features each (warps straddle two images), dead features
    interleaved, starts near all four edges and in the interior; frame pairs moved by 0.6, 2.5 and 4.5 px (the first step
    leaves the windowed kernel's 2-pixel margin: it re-stages mid-loop) and unrelated random frames."""
    f1, f2 = frames_for(motion, 3, 157, 203, seed=W * 10 + len(motion))
    step_case(gpu_ctx, f1, f2, W, windowed, "%s W%d %s" % ("windowed" if windowed else "fast", W, motion), seed=W)


def windowed_launch_shape(W, n, sms):
    """launch_windowed's choice (klt_track_windowed.cu): 4 warps per CTA when the grid is at least two waves deep."""
    fpw, minb = (2, 5) if W <= 7 else (1, 3)
    return 4 if -(-n // (4 * fpw)) >= 2 * minb * sms else 2


@gpu
@pytest.mark.parametrize("W", [7, 9])
def test_windowed_four_warp_launch(gpu_ctx, W):
    """The NW = 4 instantiation of lk_windowed (large grids: 11 840 features at 7 x 7 and 3 552 at 9 x 9 on 148 SMs) on
    1080p frames; the NW = 2 one is what every other case runs."""
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = next(n for n in range(1000, 40000, 16) if windowed_launch_shape(W, n, sms) == 4)
    assert windowed_launch_shape(W, 37 * 3, sms) == 2
    f1, f2 = frames_for("2.5px", 1, 1080, 1920, seed=W)
    step_case(gpu_ctx, f1, f2, W, True, "windowed NW4 W%d n%d" % (W, n), n_per_image=n, seed=W)


@gpu
def test_windowed_different_gradient_taps(gpu_ctx):
    """p1 built with grad_sigma 1.0 and p2 with 1.1 (both 7-tap): the windowed kernel takes its K.same == 0 path, and each
    side's reference uses its own taps."""
    t2 = taps_for(nPyramidLevels=1, subsampling=2, grad_sigma=1.1)
    assert len(t2[1].g) == 7 and len(t2[1].d) == 7
    f1, f2 = frames_for("2.5px", 3, 157, 203, seed=5)
    step_case(gpu_ctx, f1, f2, 7, True, "windowed taps 1.0 / 1.1", taps2=t2)


@gpu
@pytest.mark.parametrize("windowed", [False, True])
def test_float_images_at_level_zero(gpu_ctx, windowed):
    """Arbitrary float images in [-1000, 1000] as already-smoothed level 0 (build_f32): a FAST_WINDOWED build of it is
    image-only and the windowed tracker runs on it; the FAST build gives the row kernel its gradient planes."""
    rng = np.random.default_rng(11)
    base = rng.uniform(-1000, 1000, (3, 170, 230))
    import scipy.ndimage as ndi
    f1 = np.stack([ndi.gaussian_filter(b, 1.5)[:157, :203] for b in base]).astype(f32)
    f2 = np.stack([ndi.shift(ndi.gaussian_filter(b, 1.5), (0.7, -1.2), order=3)[:157, :203] for b in base]).astype(f32)
    step_case(gpu_ctx, np.ascontiguousarray(f1), np.ascontiguousarray(f2), 7, windowed,
              "f32 level 0 %s" % ("windowed" if windowed else "fast"), f32_input=True)


# ---- decisions: features farther than their bound from a threshold get exactly the reference's status -------------------------
def decision_setup(ctx, W, windowed, motion, seed):
    """Frames, pyramids (kept open), start positions and the retain iterates x_1, x_2 of one configuration."""
    from pyfeaturetrack_b200 import _capi
    B, H, Wd, n = 3, 157, 203, 37
    f1, f2 = frames_for(motion, B, H, Wd, seed)
    t, T = taps_for(nPyramidLevels=1, subsampling=2, window_width=W, window_height=W)
    prec = _capi.PRECISION_FAST_WINDOWED if windowed else _capi.PRECISION_FAST
    p1, p2 = _capi.Pyramid(ctx, Wd, H, 1, 2, B), _capi.Pyramid(ctx, Wd, H, 1, 2, B)
    p1.build_u8(f1, t, prec)
    p2.build_u8(f2, t, prec)
    x0, y0, v0 = start_positions(seed, B, n, W, Wd, H)
    params = make_params(W, retain_trackers=1, min_displacement=0.0)
    iters = run_iterates(ctx, params, p1, p2, n, x0, y0, v0, 2, expected_tracker(W, windowed))
    return p1, p2, T, (B, H, Wd, n), iters


DECISION_CASES = [(7, False, "2.5px"), (9, False, "4.5px"), (17, False, "2.5px"), (7, True, "2.5px"), (9, True, "4.5px"),
                  (13, True, "4.5px")]


@gpu
@pytest.mark.parametrize("W,windowed,motion", DECISION_CASES)
def test_decisions(gpu_ctx, W, windowed, motion):
    """Small determinant (min_determinant at the 25/50/75 % quantiles of the step-1 det, max_iterations 1, statuses -2 or
    -3), convergence (max_iterations 2, min_displacement at the median step-1 displacement: 0 with x_1 or -3) and residue
    (max_residue at quantiles of the residue at x_1: -5 or -3; at 4.5 px the windowed kernel re-stages for it)."""
    kind = expected_tracker(W, windowed)
    label = "%s W%d %s" % (kind, W, motion)
    p1, p2, T, (B, H, Wd, n), iters = decision_setup(gpu_ctx, W, windowed, motion, seed=W + 3)
    try:
        (x0, y0, v0, _), (x1, y1, v1, _) = iters[0], iters[1]
        # component 0 only for image-only pyramids (level_inputs): the tracks below still take lk_windowed
        lv = level_inputs(p1, p2, T, T, B, windowed)
        live = np.nonzero((v0 == 0) & ~loop_oob(x0, y0, W, Wd, H))[0]
        img = live // n
        s1 = Step(lv, img, x0[live], y0[live], x0[live], y0[live], W, kind)
        ok = s1.ok
        params = make_params(W)

        def run(**kw):
            for k, v in kw.items():
                setattr(params, k, v)
            out = []
            ran = profiled(gpu_ctx, lambda: out.append(track(gpu_ctx, params, p1, p2, n, x0, y0, v0)))
            assert tracker_of(ran) == {kind}, sorted(ran)
            return out[0]
        # x_1 of a track without retain is bit-equal to the retain track's x_1: it decides the post-loop check exactly
        post1 = post_oob(x1[live], y1[live], W, Wd, H)

        # -- small determinant: max_iterations 1, statuses -2 or -3 (-4 where x_1 fails the post-loop check)
        for q in (0.25, 0.5, 0.75):
            md = float(f32(np.quantile(s1.det[ok], q)))
            _, _, v, _ = run(max_iterations=1, min_displacement=0.1, min_determinant=md, has_max_residue=0)
            small = ok & (s1.det + s1.e_det < md)
            big = ok & (s1.det - s1.e_det >= md)
            post0 = post_oob(x0[live], y0[live], W, Wd, H)
            assert (v[live[small & ~post0]] == SMALL_DET).all() and (v[live[small & post0]] == OOB).all(), (label, q)
            assert (v[live[big & ~post1]] == MAX_ITERATIONS).all() and (v[live[big & post1]] == OOB).all(), (label, q)
            assert small.sum() > 0.15 * ok.sum() and big.sum() > 0.15 * ok.sum(), (label, q)
            print("fp64 %s min_determinant q%.2f: %d of %d decided" % (label, q, small.sum() + big.sum(), ok.sum()))
        # -- the same, with min_determinant two bounds above or below the det of the features with the tightest relative
        # bounds: a kernel det off by more than 2 e_det (a gradient tap 1e-5 off moves det by 4e-5) flips their status
        cand = np.nonzero(ok & ~post_oob(x0[live], y0[live], W, Wd, H) & ~post1)[0]
        for i in cand[np.argsort((s1.e_det / s1.det)[cand])[:3]]:
            for sign, want in ((1, SMALL_DET), (-1, MAX_ITERATIONS)):
                md = float(f32(s1.det[i] + sign * 2 * s1.e_det[i]))
                assert abs(md - s1.det[i]) > s1.e_det[i], (label, i)
                _, _, v, _ = run(max_iterations=1, min_displacement=0.1, min_determinant=md, has_max_residue=0)
                assert v[live[i]] == want, (label, i, sign, v[live[i]])
        print("fp64 %s min_determinant at 2 e_det from a det: tightest e_det / det %.2e" % (label, (s1.e_det / s1.det)[cand].min()))

        # -- convergence: max_iterations 2, min_displacement at the median step-1 displacement
        md = 0.01
        took1 = ok & (s1.det - s1.e_det >= md)
        dmax = np.maximum(np.abs(s1.dx), np.abs(s1.dy))
        e_d = np.maximum(s1.e_dx, s1.e_dy)
        th = float(f32(np.median(dmax[took1])))
        x, y, v, its = run(max_iterations=2, min_displacement=th, min_determinant=md, has_max_residue=0)
        stop = took1 & (dmax + e_d < th)
        cont = took1 & (dmax - e_d >= th)
        fs = live[stop & ~post1]
        assert (v[fs] == TRACKED).all() and np.array_equal(x[fs], x1[fs]) and np.array_equal(y[fs], y1[fs]), label
        assert (v[live[stop & post1]] == OOB).all(), label
        assert np.isin(v[live[cont]], (SMALL_DET, MAX_ITERATIONS, OOB)).all(), label
        assert stop.sum() > 0.3 * took1.sum() and cont.sum() > 0.3 * took1.sum(), label
        assert stop.sum() + cont.sum() <= its <= stop.sum() + 2 * (len(live) - stop.sum()), (label, its)
        print("fp64 %s min_displacement: %d of %d decided" % (label, stop.sum() + cont.sum(), took1.sum()))

        # -- residue at x_1 (T at x_0, P at x_1): max_iterations 1, statuses -5 or -3
        on = took1 & ~post1 & (v1[live] == TRACKED)
        lo = live[on]
        r = Step(lv, lo // n, x0[lo], y0[lo], x1[lo], y1[lo], W, kind)
        for q in (0.25, 0.5, 0.75):
            mr = float(f32(np.quantile(r.res, q)))
            _, _, v, _ = run(max_iterations=1, min_displacement=0.1, min_determinant=md, has_max_residue=1, max_residue=mr)
            big = r.res - r.e_res > mr
            small = r.res + r.e_res <= mr
            assert (v[lo[big]] == LARGE_RESIDUE).all() and (v[lo[small]] == MAX_ITERATIONS).all(), (label, q)
            assert big.sum() > 0.15 * len(lo) and small.sum() > 0.15 * len(lo), (label, q)
            print("fp64 %s max_residue q%.2f: %d of %d decided" % (label, q, big.sum() + small.sum(), on.sum()))
    finally:
        p1.close(); p2.close()


def static_track(x0, y0, W, L, ss, dims, bx, by):
    """What a track does on identical frames (diff == 0, so every step is exactly 0): ('assert', ...) or (status, x, y,
    iterations), restating the level loop, its checks and the final border check in the kernels' arithmetic."""
    xloc, yloc = x0, y0
    for _ in range(L):
        xloc, yloc = xloc / ss, yloc / ss
    xout, yout = xloc, yloc
    its, status = 0, TRACKED
    for r in range(L - 1, -1, -1):
        xloc, yloc, xout, yout = xloc * ss, yloc * ss, xout * ss, yout * ss
        nc, nr = dims[r]
        if template_assert(xloc, yloc, W, nc, nr):
            return "assert", r
        x2, y2 = f32(xout), f32(yout)
        status = OOB if loop_oob(x2, y2, W, nc, nr) else TRACKED
        its += status == TRACKED
        if post_oob(x2, y2, W, nc, nr):
            status = OOB
        xout, yout = float(x2), float(y2)
        if status == OOB:
            break
    W0, H0 = dims[0]
    if status == OOB or border_oob(xout, yout, W0, H0, bx, by):
        return OOB, -1.0, -1.0, its
    return TRACKED, xout, yout, its


def border_probes(W, ss, dims, bx):
    """Positions on both sides of every threshold at every level r (x / ss**r): left, the in-loop check (integer hw) and
    the template assertion (both at hw), the post-loop check at hw + 0.5; right, the in-loop check at n - hw - 1.001, the
    assertion at n - hw - 1, the post-loop check at n - hw - 1.501; and the final border bx on both sides at level 0.  One
    coordinate probes, the other sits in the middle of the image.  Dyadic values: exact at every level."""
    hw, probes = W // 2, []
    for r in range(len(dims)):
        for axis, n in ((0, dims[r][0]), (1, dims[r][1])):
            for v in (hw, hw - 2 ** -8, hw + 0.5 - 2 ** -9, hw + 0.5 + 2 ** -9, n - hw - 1 - 2 ** -9, n - hw - 1 - 2 ** -11,
                      n - hw - 1, n - hw - 1.5 - 2 ** -9, n - hw - 1.5 - 2 ** -11):
                probes.append((axis, v * ss ** r))
    for axis, n in ((0, dims[0][0]), (1, dims[0][1])):
        for v in (bx - 2 ** -9, bx + 2 ** -9, n - 1 - bx - 2 ** -9, n - 1 - bx + 2 ** -9):
            probes.append((axis, v))
    cx, cy = float(dims[0][0] // 2), float(dims[0][1] // 2)
    return np.array([v if a == 0 else cx for a, v in probes]), np.array([v if a == 1 else cy for a, v in probes])


@pytest.mark.parametrize("L", [1, 2])
@pytest.mark.parametrize("W", [7, 17])
def test_static_track_matches_oracle(oracle, W, L):
    """static_track against oracle.track_on_pyramids on identical frames at every border probe: the same assertion,
    status, position and iteration count."""
    H, Wd, ss, bx = 157, 203, 2, 20.5
    frame = frames_for("0.6px", 1, H, Wd, seed=W + L)[0][0]
    p = oracle.Params(window_width=W, window_height=W, nPyramidLevels=L, subsampling=ss, min_determinant=-1.0)
    p.borderx = p.bordery = bx
    pyr = oracle.image_pyramids(p, frame)
    dims = [(a.shape[1], a.shape[0]) for a in pyr[0]]
    kinds = set()
    for x, y in zip(*border_probes(W, ss, dims, bx)):
        want = static_track(x, y, W, L, ss, dims, bx, bx)
        kinds.add(want[0])
        if want[0] == "assert":
            with pytest.raises(AssertionError):
                oracle.track_on_pyramids(p, pyr, pyr, [x], [y], [0])
            continue
        gx, gy, gv, its = oracle.track_on_pyramids(p, pyr, pyr, [x], [y], [0])
        assert (gv[0], gx[0], gy[0], its) == want, (x, y)
    assert kinds == {TRACKED, OOB, "assert"}


@gpu
@pytest.mark.parametrize("L", [1, 2])
@pytest.mark.parametrize("W,windowed", [(7, False), (17, False), (7, True), (11, True)])
def test_borders_and_assertions_on_identical_frames(gpu_ctx, W, windowed, L):
    """Identical frames make diff == 0, so d == 0 exactly and positions stay where the test put them.  Positions on both
    sides of every threshold, at every level (x / ss**r): the float in-loop check with integer hw, the double post-loop check
    with W / 2.0, the final border check and the template assertion.  Positions that assert go in calls of their own, which
    return KLT_ERR_ASSERT and leave the lists untouched; the others get exactly the restated status, position and
    iteration count."""
    from pyfeaturetrack_b200 import _capi
    H, Wd, ss, bx = 157, 203, 2, 20.5
    frame = frames_for("0.6px", 1, H, Wd, seed=W + L)[0]
    t, _ = taps_for(nPyramidLevels=L, subsampling=ss, window_width=W, window_height=W)
    prec = _capi.PRECISION_FAST_WINDOWED if windowed else _capi.PRECISION_FAST
    p1, p2 = _capi.Pyramid(gpu_ctx, Wd, H, L, ss, 1), _capi.Pyramid(gpu_ctx, Wd, H, L, ss, 1)
    try:
        p1.build_u8(frame, t, prec)
        p2.build_u8(frame, t, prec)
        dims = [d[:2] for d in p1.dims]
        xs, ys = border_probes(W, ss, dims, bx)
        want = [static_track(x, y, W, L, ss, dims, bx, bx) for x, y in zip(xs, ys)]
        asserts = np.array([w[0] == "assert" for w in want])
        assert asserts.sum() >= 4 * L and {w[0] for w in want} >= {TRACKED, OOB, "assert"}
        params = make_params(W, L=L, ss=ss, borderx=bx, bordery=bx, min_determinant=-1.0)
        kind = expected_tracker(W, windowed)
        lib = _capi.lib()
        for f in np.nonzero(asserts)[0]:
            x, y, v = xs[f:f + 1].copy(), ys[f:f + 1].copy(), np.zeros(1, np.int32)
            with pytest.raises(AssertionError):
                gpu_ctx.check(lib.klt_track_features(gpu_ctx.handle, C.byref(params), p1.handle, p2.handle, 1, x.ctypes.data,
                                                     y.ctypes.data, v.ctypes.data, None))
            assert x[0] == xs[f] and y[0] == ys[f] and v[0] == 0, (xs[f], ys[f])
        keep = ~asserts
        n = int(keep.sum())
        out = []
        ran = profiled(gpu_ctx, lambda: out.append(track(gpu_ctx, params, p1, p2, n, xs[keep], ys[keep], np.zeros(n, np.int32))))
        assert tracker_of(ran) == {kind}, sorted(ran)
        x, y, v, its = out[0]
        ws = [w for w in want if w[0] != "assert"]
        assert list(v) == [w[0] for w in ws], list(zip(xs[keep], ys[keep], v, [w[0] for w in ws]))
        assert np.array_equal(x, [w[1] for w in ws]) and np.array_equal(y, [w[2] for w in ws])
        assert its == sum(w[3] for w in ws)
        print("fp64 %s W%d L%d borders: %d positions, %d asserting, statuses %s" % (kind, W, L, len(want), asserts.sum(),
                                                                                  np.unique(v, return_counts=True)))
    finally:
        p1.close(); p2.close()


# ---- several levels, end to end: the per-level tensor maps, offsets and pitches -------------------------------------------------
def chain_reference(lvs, dims, x0, y0, img, W, L, ss, kind, n_steps, min_det, e_max=1e-4):
    """The float64 chain of a retain track with min_displacement 0 and max_iterations = n_steps, from the coarsest level
    down.  Its error bound is propagated per step as E <- 2 ||J||_inf E + b, J the central-difference Jacobian of the float64
    step map at the reference iterate (h = 1e-3 px, the worse of the one-sided values), b the step's own bound, and scaled
    by ss between levels.  Returns (x, y, E, kept): kept drops features whose E exceeds e_max or whose checks (in-loop and
    post-loop, small determinant, conditioning) are not decided by the bound."""
    h = 1e-3
    act = np.arange(len(x0))
    xl, yl = np.asarray(x0, np.float64) / ss ** L, np.asarray(y0, np.float64) / ss ** L
    xr, yr, E = xl.copy(), yl.copy(), np.zeros(len(x0))
    for r in range(L - 1, -1, -1):
        xl, yl, xr, yr, E = xl * ss, yl * ss, xr * ss, yr * ss, E * ss
        nc, nr = dims[r]
        x1, y1 = f32(xl).astype(np.float64), f32(yl).astype(np.float64)
        for _ in range(n_steps):
            a = act
            corners = [loop_oob(xr[a] + sx * E[a], yr[a] + sy * E[a], W, nc, nr) for sx in (-1, 1) for sy in (-1, 1)]
            act = a[~np.any(corners, axis=0)]
            a = act
            s = Step(lvs[r], img[a], x1[a], y1[a], xr[a], yr[a], W, kind)
            J = np.zeros((len(a), 2, 2))
            for j, (hx, hy) in enumerate(((h, 0), (0, h))):
                up = Step(lvs[r], img[a], x1[a], y1[a], xr[a] + hx, yr[a] + hy, W, kind)
                dn = Step(lvs[r], img[a], x1[a], y1[a], xr[a] - hx, yr[a] - hy, W, kind)
                J[:, 0, j] = np.maximum(np.abs(up.x - s.x), np.abs(s.x - dn.x)) / h
                J[:, 1, j] = np.maximum(np.abs(up.y - s.y), np.abs(s.y - dn.y)) / h
            Jn = np.abs(J).sum(2).max(1)
            E[a] = 2 * Jn * E[a] + np.maximum(s.e_x, s.e_y)
            xr[a], yr[a] = s.x, s.y
            keep = s.ok & (s.det - s.e_det >= min_det) & (E[a] <= e_max)
            act = a[keep]
        a = act
        corners = [post_oob(xr[a] + sx * E[a], yr[a] + sy * E[a], W, nc, nr) for sx in (-1, 1) for sy in (-1, 1)]
        act = a[~np.any(corners, axis=0)]
    kept = np.zeros(len(x0), bool)
    kept[act] = True
    return xr, yr, E, kept


def rough_pairs(seed, B, H, W, shift):
    """Random u8 frames and the same moved by `shift` (cubic, rounded back to u8): gradients of tens of units per pixel,
    which keep the propagated bound of a multi-level chain small."""
    import scipy.ndimage as ndi
    f1 = random_frames(seed, B, H, W)
    f2 = np.stack([np.clip(np.rint(ndi.shift(f.astype(np.float64), shift, order=3, mode="reflect")), 0, 255) for f in f1])
    return f1, f2.astype(np.uint8)


@pytest.mark.parametrize("W,L,ss", [(7, 3, 2), (17, 2, 4)])
def test_chain_reference_matches_oracle(oracle, W, L, ss):
    """chain_reference with the exact-order bound against oracle.track_on_pyramids through every level: the oracle's
    positions lie within the propagated bound of every feature the chain keeps (any bound here: this pins the chain,
    not its sensitivity)."""
    H, Wd, n = 300, 400, 60
    p = oracle.Params(window_width=W, window_height=W, nPyramidLevels=L, subsampling=ss, retainTrackers=True,
                      min_displacement=0.0, max_iterations=3)
    p.borderx = p.bordery = 0.0
    f1, f2 = rough_pairs(W + L, 1, H, Wd, (-1.5, 2.5))
    a, b = oracle.image_pyramids(p, f1[0]), oracle.image_pyramids(p, f2[0])
    lvs = [Level(*(c[lvl][None].astype(np.float64) for c in a), [0.0], *(c[lvl][None].astype(np.float64) for c in b), [0.0])
           for lvl in range(L)]
    dims = [(lv.shape[1], lv.shape[0]) for lv in a[0]]
    x0, y0 = interior_starts(np.random.default_rng(W), n, W, Wd, H, (W // 2 + 6) * ss ** (L - 1))
    x, y, v, _ = oracle.track_on_pyramids(p, a, b, x0, y0, np.zeros(n, np.int32))
    xr, yr, E, kept = chain_reference(lvs, dims, x0, y0, np.zeros(n, np.int64), W, L, ss, "lk_track", 3, p.min_determinant,
                                      e_max=1.0)
    assert (v[kept] == TRACKED).all() and kept.sum() >= 0.9 * n
    record("lk_track oracle levels", np.abs(x[kept] - xr[kept]), E[kept], "oracle W%d L%d ss%d x" % (W, L, ss))
    record("lk_track oracle levels", np.abs(y[kept] - yr[kept]), E[kept], "oracle W%d L%d ss%d y" % (W, L, ss))


@gpu
@pytest.mark.parametrize("L,ss", [(3, 2), (2, 4)])
@pytest.mark.parametrize("W,windowed", [(7, False), (15, False), (7, True), (11, True)])
def test_pyramid_levels_end_to_end(gpu_ctx, W, windowed, L, ss):
    """Retain tracks with min_displacement 0 and max_iterations 3 through L = 3, ss = 2 and L = 2, ss = 4 on a batch of two
    300 x 400 random frames moved by (-1.5, 2.5) px, against the float64 chain with its propagated bound: the only cases
    that read levels >= 1, through the per-level tensor maps, plane offsets and pitches."""
    from pyfeaturetrack_b200 import _capi
    B, H, Wd, n, steps = 2, 300, 400, 37, 3
    kind = expected_tracker(W, windowed)
    label = "%s W%d L%d ss%d" % (kind, W, L, ss)
    f1, f2 = rough_pairs(W * L + ss, B, H, Wd, (-1.5, 2.5))
    t, T = taps_for(nPyramidLevels=L, subsampling=ss, window_width=W, window_height=W)
    prec = _capi.PRECISION_FAST_WINDOWED if windowed else _capi.PRECISION_FAST
    p1, p2 = _capi.Pyramid(gpu_ctx, Wd, H, L, ss, B), _capi.Pyramid(gpu_ctx, Wd, H, L, ss, B)
    try:
        p1.build_u8(f1, t, prec)
        p2.build_u8(f2, t, prec)
        rng = np.random.default_rng(W + L)
        x0, y0 = interior_starts(rng, B * n, W, Wd, H, (W // 2 + 6) * ss ** (L - 1))
        v0 = np.where(np.arange(B * n) % 8 == 7, -1, 0).astype(np.int32)
        params = make_params(W, L=L, ss=ss, retain_trackers=1, min_displacement=0.0, max_iterations=steps)
        out = []
        ran = profiled(gpu_ctx, lambda: out.append(track(gpu_ctx, params, p1, p2, n, x0, y0, v0)))
        assert tracker_of(ran) == {kind}, sorted(ran)
        x, y, v, _ = out[0]
        lvs = [level_inputs(p1, p2, T, T, B, windowed, lvl) for lvl in range(L)]
        dims = [d[:2] for d in p1.dims]
    finally:
        p1.close(); p2.close()
    dead = v0 < 0
    assert np.array_equal(x[dead], x0[dead]) and np.array_equal(v[dead], v0[dead])
    img = np.arange(B * n) // n
    # 1e-3 px: three Newton steps per level do not contract the coarse levels' bounds (times ss per level) much below
    # 1e-4 px, and a wrong level offset, pitch or tensor map moves a position by pixels
    xr, yr, E, kept = chain_reference(lvs, dims, x0, y0, img, W, L, ss, kind, steps, params.min_determinant, e_max=1e-3)
    kept &= ~dead
    assert (v[kept] == TRACKED).all(), label
    record(kind + " levels", np.abs(x[kept] - xr[kept]), E[kept], label + " x")
    record(kind + " levels", np.abs(y[kept] - yr[kept]), E[kept], label + " y")
    print("fp64 %s: %d of %d live features checked end to end (%d with a bound under 1e-4 px), median propagated bound "
          "%.3e px" % (label, kept.sum(), (~dead).sum(), (kept & (E <= 1e-4)).sum(), np.median(E[kept])))
    assert kept.sum() >= 0.25 * (~dead).sum(), label
