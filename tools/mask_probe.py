"""Cost of a selection mask, device-timed.  Prints one JSON line per measurement, each with the GPU's name and power limit.

  python tools/mask_probe.py               sequence step (8 x 1080p x 1000 features, windowed tracking, fast selection) with
                                           no mask, an all-ones mask (same lists as no mask: the cost of the mechanism alone),
                                           a fixed mask, and a mask replaced before every step; and a batched fast selection of
                                           64 device-resident 1080p frames without a mask, with an all-ones and with a per-frame
                                           mask.
                                           Variants alternate, three rounds, one process
  python tools/mask_probe.py --profile     per-kernel split of the same workloads from the launch profile (separate run)
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


def make_masks(count, H, W, seed=0):
    """A black border, a burned-in block and about a quarter of 32-px cells masked out, different per frame."""
    rng = np.random.default_rng(seed)
    out = np.ones((count, H, W), np.uint8)
    for i in range(count):
        cells = rng.random(((H + 31) // 32, (W + 31) // 32)) >= 0.25
        out[i] = np.kron(cells, np.ones((32, 32), np.uint8))[:H, :W]
        out[i, :40] = out[i, -40:] = 0
        out[i, :, :40] = out[i, :, -40:] = 0
        out[i, 60:120, 1400:1860] = 0
    return out


def sequence_leg(ctx, args, info, profile=False):
    """ms per klt_sequence step (B x 1080p, n features, FAST_WINDOWED + SELECT_FAST, device frames, graphs): no mask, one
    all-ones device mask, a fixed per-sequence device mask, and a device mask replaced (klt_sequence_set_mask) before every
    step."""
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
    masks = make_masks(2 * B, H, W, seed=1)
    dmask = ctx.device_alloc(masks.nbytes)
    ctx.memcpy(dmask, masks, masks.nbytes)
    dones = ctx.device_alloc(H * W)
    ctx.memcpy(dones, np.ones((H, W), np.uint8), H * W)
    ctx.sync()
    per, mper = B * H * W, H * W
    modes = ["off", "ones", "fixed", "per_step"]
    seqs = {}

    def step(m, q, k):
        if m == "per_step":
            q.set_mask(dmask + (k % 2) * B * mper, W, mper)
        q.step(dfr + (k % distinct) * per)
    for m in modes:
        q = _capi.Sequence(ctx, params, taps, W, H, B, n, _capi.PRECISION_FAST_WINDOWED, _capi.SELECT_FAST)
        if m == "ones":
            q.set_mask(dones, W, 0)
        elif m != "off":
            q.set_mask(dmask, W, mper)
        q.start(dfr)
        for k in range(1, 9):                        # warm-up: plain launches, then graph capture for every rotation slot
            step(m, q, k)
        q.sync()
        seqs[m] = [q, 9]
    if profile:
        out = {}
        for m in modes:
            ctx.profile(True)
            ctx.profile_reset()
            q, k0 = seqs[m]
            for k in range(args.steps):
                step(m, q, k0 + k)
            q.sync()
            out[m] = {k: dict(ms_per_step=round(v["ms"] / args.steps, 5), launches=v["launches"])
                      for k, v in sorted(ctx.profile_read().items())}
            ctx.profile(False)
            seqs[m][1] = k0 + args.steps
        print(json.dumps(dict(info, leg="sequence_profile", B=B, n=n, steps=args.steps, kernels=out)))
    else:
        times = {m: [] for m in modes}
        for r in range(args.rounds):
            for m in modes:
                q, k0 = seqs[m]
                ctx.timer_start()
                for k in range(args.steps):
                    step(m, q, k0 + k)
                ctx.timer_stop()
                times[m].append(ctx.timer_elapsed_ms() / args.steps)
                q.sync()
                seqs[m][1] = k0 + args.steps
        res = dict(info, leg="sequence_step", B=B, n=n, steps_per_round=args.steps,
                   graphs={m: seqs[m][0].uses_graph() for m in modes})
        for m in modes:
            res["%s_ms" % m] = [round(t, 4) for t in times[m]]
        for m in modes[1:]:
            res["added_ms_per_step_%s" % m] = round(float(np.median(times[m]) - np.median(times["off"])), 4)
        for m in ("off", "ones"):
            res["%s_lists_after_%d_steps" % (m, seqs[m][1])] = digest(*seqs[m][0].features())
        print(json.dumps(res))
    sys.stdout.flush()
    for q, _ in seqs.values():
        q.close()
    ctx.device_free(dfr)
    ctx.device_free(dmask)
    ctx.device_free(dones)
    ctx.free_pinned(frames)


def batch_leg(ctx, args, info, profile=False):
    """klt_select_good_features_batch(_masked) (SELECT_FAST) on one 64-frame 1080p image-only pyramid built once, device lists,
    nothing waits; one all-ones mask (stride 0), or a different device mask per frame."""
    from pyfeaturetrack_b200 import _capi, klt, synth, selectGoodFeatures as sgf, trackFeatures as tf
    tc = make_tc(klt)
    tc.sequentialMode = False
    params, taps = sgf.make_params(tc), tf._taps_for_one_image(tc)
    H, W, P, n = 1080, 1920, 64, args.n
    base = synth.fast_frames(H, W, 16, seed=3)
    pyr = _capi.Pyramid(ctx, W, H, 3, 2, P)
    pyr.build_u8(np.ascontiguousarray(np.stack([base[i % 16] for i in range(P)])), taps, _capi.PRECISION_FAST_WINDOWED)
    masks = make_masks(P, H, W, seed=2)
    dmask = ctx.device_alloc(masks.nbytes)
    ctx.memcpy(dmask, masks, masks.nbytes)
    dones = ctx.device_alloc(H * W)
    ctx.memcpy(dones, np.ones((H, W), np.uint8), H * W)
    dl = [ctx.device_alloc(P * n * 8), ctx.device_alloc(P * n * 8), ctx.device_alloc(P * n * 4)]
    ctx.sync()
    lib = _capi.lib()

    def call(m):
        if m == "off":
            ctx.check(lib.klt_select_good_features_batch(ctx.handle, C.byref(params), pyr.handle, n, 0, _capi.SELECT_FAST,
                                                         dl[0], dl[1], dl[2]))
        else:
            mp, stride = (dones, 0) if m == "ones" else (dmask, H * W)
            ctx.check(lib.klt_select_good_features_batch_masked(ctx.handle, C.byref(params), pyr.handle, n, 0, _capi.SELECT_FAST,
                                                                mp, W, stride, dl[0], dl[1], dl[2]))
    modes = ["off", "ones", "masked"]
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
            out[m] = {k: dict(ms_per_call=round(val["ms"] / args.calls, 5), launches=val["launches"])
                      for k, val in sorted(ctx.profile_read().items())}
            ctx.profile(False)
        print(json.dumps(dict(info, leg="batch_profile", frames=P, n=n, calls=args.calls, kernels=out)))
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
        res = dict(info, leg="batch_select_64", frames=P, n=n, calls_per_round=args.calls)
        for m in modes:
            res["%s_ms" % m] = [round(t, 4) for t in times[m]]
        for m in modes[1:]:
            res["added_ms_per_call_%s" % m] = round(float(np.median(times[m]) - np.median(times["off"])), 4)
        print(json.dumps(res))
    sys.stdout.flush()
    for d in dl + [dmask, dones]:
        ctx.device_free(d)
    pyr.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--B", type=int, default=8)
    ap.add_argument("--n", type=int, default=1000)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--calls", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--legs", default="sequence,batch")
    args = ap.parse_args()
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from pyfeaturetrack_b200 import _capi
    ctx = _capi.Context(0)
    info = gpu_info()
    for leg in args.legs.split(","):
        {"sequence": sequence_leg, "batch": batch_leg}[leg](ctx, args, info, profile=args.profile)
    ctx.close()


if __name__ == "__main__":
    main()
