"""Cost of the forward-backward check, device-timed.  Prints one JSON line per measurement, each with the GPU's name and power
limit.

  python tools/fb_probe.py                 sequence step (8 x 1080p x 1000 features, windowed tracking, fast selection) and
                                           klt_track_features_fb against klt_track_features on 64 device-resident config-B
                                           pairs: FB off and FB on alternating, three rounds, one process
  python tools/fb_probe.py --profile       per-kernel split of the same two workloads from the launch profile (separate run)
  python tools/fb_probe.py --off-only      FB off only, plus a digest of the resulting lists: runs against a tree without the
                                           check (--tree), to compare step time and results with it in the same session
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:           # noqa: BLE001 -- the numbers stay valid, only their label is missing
        return {"gpu": "unknown (%s)" % e, "power_limit": "unknown"}


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def make_tc(klt):
    tc = klt.KLT_TrackingContext()
    tc.nPyramidLevels, tc.subsampling, tc.max_residue, tc.sequentialMode = 3, 2, 10.0, True
    tc.KLTUpdateTCBorder()
    return tc


def sequence_leg(ctx, args, fb, info, profile=False):
    """ms per klt_sequence step (B x 1080p, n features, FAST_WINDOWED + SELECT_FAST, device frames, graphs) with the check off
    (fb = None) or on at `fb` px; rounds alternate the two sequences."""
    from pyfeaturetrack_b200 import _capi, klt, synth, selectGoodFeatures as sgf, trackFeatures as tf
    tc = make_tc(klt)
    params, taps = sgf.make_params(tc), tf._taps_for_one_image(tc)
    H, W, B, n, distinct = 1080, 1920, args.B, args.n, 16
    base = [synth.fast_frames(H, W, distinct, seed=7 + s) for s in range(4)]
    frames = ctx.pinned_array((distinct, B, H, W), np.uint8)
    for k in range(distinct):
        for s in range(B):
            frames[k, s] = base[s % 4][(k + s // 4) % distinct]
    dfr = ctx.device_alloc(frames.nbytes)
    ctx.memcpy(dfr, frames, frames.nbytes)
    ctx.sync()
    per = B * H * W
    modes = [None] if fb is None else [None, fb]
    seqs = {}
    for m in modes:
        q = _capi.Sequence(ctx, params, taps, W, H, B, n, _capi.PRECISION_FAST_WINDOWED, _capi.SELECT_FAST)
        q.start(dfr)
        if m is not None:
            q.set_fb_check(m)
        for k in range(1, 9):                        # warm-up: plain launches, then graph capture for every rotation slot
            q.step(dfr + (k % distinct) * per)
        q.sync()
        seqs[m] = [q, 9]
    if profile:
        out = {}
        for m in modes:
            ctx.profile(True)
            ctx.profile_reset()
            q, k0 = seqs[m]
            for k in range(args.steps):
                q.step(dfr + ((k0 + k) % distinct) * per)
            q.sync()
            out["fb_on" if m else "fb_off"] = {k: dict(ms_per_step=round(v["ms"] / args.steps, 5), launches=v["launches"])
                                               for k, v in sorted(ctx.profile_read().items())}
            ctx.profile(False)
        print(json.dumps(dict(info, leg="sequence_profile", B=B, n=n, steps=args.steps, kernels=out)))
        sys.stdout.flush()
    else:
        times = {m: [] for m in modes}
        for r in range(args.rounds):
            for m in modes:
                q, k0 = seqs[m]
                ctx.timer_start()
                for k in range(args.steps):
                    q.step(dfr + ((k0 + k) % distinct) * per)
                ctx.timer_stop()
                times[m].append(ctx.timer_elapsed_ms() / args.steps)
                q.sync()
                seqs[m][1] = k0 + args.steps
        res = dict(info, leg="sequence_step", B=B, n=n, steps_per_round=args.steps,
                   fb_off_ms=[round(t, 4) for t in times[None]])
        if fb is not None:
            res["fb_on_ms"] = [round(t, 4) for t in times[fb]]
            res["fb_max_error_px"] = fb
            res["added_ms_per_step"] = round(float(np.median(times[fb]) - np.median(times[None])), 4)
        x, y, v, vt = seqs[None][0].features()
        res["fb_off_lists_after_%d_steps" % seqs[None][1]] = digest(x, y, v, vt)
        print(json.dumps(res))
        sys.stdout.flush()
    for q, _ in seqs.values():
        q.close()
    ctx.device_free(dfr)
    ctx.free_pinned(frames)


def pairs_leg(ctx, args, fb, info, profile=False):
    """klt_track_features (fb None) / klt_track_features_fb on 64 device-resident config-B pairs (1080p, 1000 features, image-only
    pyramids built once), device arrays without n_iterations (nothing waits); x, y, val reset by a device copy before every call."""
    from pyfeaturetrack_b200 import _capi, klt, synth, selectGoodFeatures as sgf, trackFeatures as tf
    tc = make_tc(klt)
    tc.sequentialMode = False
    params, taps = sgf.make_params(tc), tf._taps_for_one_image(tc)
    H, W, P, n = 1080, 1920, 64, 1000
    f1, f2 = synth.frame_pair(H, W, seed=0)
    pyr1, pyr2 = _capi.Pyramid(ctx, W, H, 3, 2, P), _capi.Pyramid(ctx, W, H, 3, 2, P)
    pyr1.build_u8(np.ascontiguousarray(np.broadcast_to(f1, (P, H, W))), taps, _capi.PRECISION_FAST_WINDOWED)
    pyr2.build_u8(np.ascontiguousarray(np.broadcast_to(f2, (P, H, W))), taps, _capi.PRECISION_FAST_WINDOWED)
    sp = _capi.Pyramid(ctx, W, H, 3, 2, 1)
    sp.build_u8(np.ascontiguousarray(f1), taps, _capi.PRECISION_STRICT)
    x = np.full((P, n), -1.0); y = np.full((P, n), -1.0); v = np.full((P, n), -1, np.int32)
    ctx.check(_capi.lib().klt_select_good_features(ctx.handle, C.byref(params), sp.handle, 0, None, None, 0, 0, n, 0,
                                                   x[0].ctypes.data, y[0].ctypes.data, v[0].ctypes.data, None))
    x[:], y[:], v[:] = x[0], y[0], v[0]
    src = [ctx.device_alloc(a.nbytes) for a in (x, y, v)]
    dst = [ctx.device_alloc(a.nbytes) for a in (x, y, v)]
    for d, a in zip(src, (x, y, v)):
        ctx.memcpy(d, a, a.nbytes)
    ctx.sync()
    lib = _capi.lib()

    def call(m):
        for d, s_, a in zip(dst, src, (x, y, v)):
            ctx.memcpy(d, s_, a.nbytes)
        if m is None:
            ctx.check(lib.klt_track_features(ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, n, dst[0], dst[1], dst[2], None))
        else:
            ctx.check(lib.klt_track_features_fb(ctx.handle, C.byref(params), pyr1.handle, pyr2.handle, n, m, dst[0], dst[1],
                                                dst[2], None, None))
    modes = [None] if fb is None else [None, fb]
    for m in modes:
        for _ in range(3):
            call(m)
    ctx.sync()
    if profile:
        out = {}
        for m in modes:
            ctx.profile(True)
            ctx.profile_reset()
            for _ in range(args.calls):
                call(m)
            ctx.sync()
            out["fb_on" if m else "fb_off"] = {k: dict(ms_per_call=round(val["ms"] / args.calls, 5), launches=val["launches"])
                                               for k, val in sorted(ctx.profile_read().items())}
            ctx.profile(False)
        print(json.dumps(dict(info, leg="pairs_profile", pairs=P, n=n, calls=args.calls, kernels=out)))
    else:
        times = {m: [] for m in modes}
        for r in range(args.rounds):
            for m in modes:
                ctx.timer_start()
                for _ in range(args.calls):
                    call(m)
                ctx.timer_stop()
                times[m].append(ctx.timer_elapsed_ms() / args.calls)
                ctx.sync()
        res = dict(info, leg="pairs_64", pairs=P, n=n, calls_per_round=args.calls, note="includes 3 device copies per call",
                   fb_off_ms=[round(t, 4) for t in times[None]])
        if fb is not None:
            res["fb_on_ms"] = [round(t, 4) for t in times[fb]]
            res["fb_max_error_px"] = fb
            res["added_ms_per_64_pairs"] = round(float(np.median(times[fb]) - np.median(times[None])), 4)
            call(fb)
            vv = np.empty_like(v)
            ctx.memcpy(vv, dst[2], vv.nbytes)
            ctx.sync()
            res["fb_rejected"] = int((vv == -6).sum())
        print(json.dumps(res))
    sys.stdout.flush()
    for d in src + dst:
        ctx.device_free(d)
    for p_ in (pyr1, pyr2, sp):
        p_.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                    help="repository tree whose pyfeaturetrack_b200 is measured")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--off-only", action="store_true")
    ap.add_argument("--fb", type=float, default=1.0, help="max_fb_error of the FB-on runs (px)")
    ap.add_argument("--B", type=int, default=8)
    ap.add_argument("--n", type=int, default=1000)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--calls", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--legs", default="sequence,pairs")
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.tree))
    from pyfeaturetrack_b200 import _capi
    ctx = _capi.Context(0)
    info = dict(gpu_info(), tree=os.path.abspath(args.tree))
    fb = None if args.off_only else args.fb
    for leg in args.legs.split(","):
        {"sequence": sequence_leg, "pairs": pairs_leg}[leg](ctx, args, fb, info, profile=args.profile)
    ctx.close()


if __name__ == "__main__":
    main()
