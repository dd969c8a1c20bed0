"""Pyramid-build probe: per-kernel CUDA-event times of image-only (windowed) and dense (fast) builds for several batch
sizes, plus checksums of the built levels, so that two builds of the library can be compared kernel by kernel.
python tools/build_probe.py [--batches 8,64] [--reps 20]"""
import argparse
import json
import os
import sys
import zlib

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="8,64")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--H", type=int, default=1080)
    ap.add_argument("--W", type=int, default=1920)
    ap.add_argument("--levels", type=int, default=3)
    ap.add_argument("--modes", default="windowed")
    args = ap.parse_args()
    from pyfeaturetrack_b200 import _capi, klt, synth, trackFeatures as tf
    ctx = _capi.default_ctx()
    tc = klt.KLT_TrackingContext()
    tc.nPyramidLevels, tc.subsampling = args.levels, 2
    tc.KLTUpdateTCBorder()
    taps = tf._taps_for_one_image(tc)
    peak = 6553.0
    try:
        peak = float(json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    H, W = args.H, args.W
    base = synth.fast_frames(H, W, 4, seed=3)
    for B in [int(b) for b in args.batches.split(",")]:
        frames = np.stack([base[i % 4] for i in range(B)])
        dfr = ctx.device_alloc(frames.nbytes)
        ctx.memcpy(dfr, frames, frames.nbytes)
        ctx.sync()
        for mode in args.modes.split(","):
            prec = {"windowed": _capi.PRECISION_FAST_WINDOWED, "fast": _capi.PRECISION_FAST}[mode]
            pyr = _capi.Pyramid(ctx, W, H, args.levels, 2, batch=B)
            for _ in range(3):
                pyr.build_u8(dfr, taps, prec, pitch=W, frame_stride=W * H)
            ctx.sync()
            ctx.profile(True)
            ctx.profile_reset()
            for _ in range(args.reps):
                pyr.build_u8(dfr, taps, prec, pitch=W, frame_stride=W * H)
            ctx.sync()
            prof = ctx.profile_read()
            ctx.profile(False)
            ctx.timer_start()
            for _ in range(args.reps):
                pyr.build_u8(dfr, taps, prec, pitch=W, frame_stride=W * H)
            ctx.timer_stop()
            ms_build = ctx.timer_elapsed_ms() / args.reps
            crc = [zlib.crc32(pyr.download(0, l, image=B - 1).tobytes()) for l in range(args.levels)]
            lv = [pyr.download(0, l, image=B - 1) for l in range(args.levels)]
            rec = {"batch": B, "mode": mode, "image": "%dx%d" % (W, H), "ms_per_build": round(ms_build, 4),
                   "frames_per_s": round(B / ms_build * 1e3, 1), "crc_levels": crc,
                   "level_sums": [float(np.float64(a.sum(dtype=np.float64))) for a in lv]}
            for k, v in prof.items():
                ms = v["ms"] / v["launches"]
                gbps = v["bytes"] / v["launches"] / ms * 1e-6
                rec[k] = {"ms_per_launch": round(ms, 5), "launches": v["launches"] // args.reps, "gbps": round(gbps, 1),
                          "frac": round(gbps / peak, 4)}
            print(json.dumps(rec), flush=True)
            pyr.close()
        ctx.device_free(dfr)


if __name__ == "__main__":
    main()
