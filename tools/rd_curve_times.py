"""Rate-distortion timings: pxz_rd_curve, pxz_shrink_to_error for three PSNR targets, and pxz_shrink at the chosen factor.
    python tools/rd_curve_times.py [reps] [--out FILE]

Frames: bench.py's synthetic 8K RGBA frame and a 32768^2 RGBA frame of the same generator, made on the device; 64x64
blocks, Lanczos3 down and up, both metrics.  Wall times come from a host clock around the call and a stream synchronise
(median of `reps` calls after one warm-up; the 32768^2 frame runs max(1, reps // 3) calls); device times from the library's
per-launch events (pxz_profile_*), mean per call, for the curve call.  CUB's sort and scans count as one launch each."""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import pixlzr_b200 as P  # noqa: E402

N = P.native
args = [a for a in sys.argv[1:] if not a.startswith("--")]
REPS = int(args[0]) if args else 5
OUT = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
BS, LZ = 64, int(P.FilterType.Lanczos3)
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"(nvidia-smi not readable: {e})"
    return q


def timed(ctx, fn, reps):
    """(wall ms median, {profile name: (device ms per call, launches per call)}) over reps calls after one warm-up"""
    fn()
    ctx.synchronize()
    ctx.profile_enable(True)
    walls = []
    for _ in range(reps):
        t = time.perf_counter()
        fn()
        ctx.synchronize()
        walls.append((time.perf_counter() - t) * 1e3)
    prof = ctx.profile_read()
    ctx.profile_enable(False)
    return float(np.median(walls)), {k: (ms / reps, n / reps) for k, (ms, n) in prof.items() if n}


def frame_table(ctx, img, label, reps):
    samples = img.w * img.h * img.c
    for mname, metric in (("Oklab-MAD", N.METRIC_OKLAB_MAD), ("Sobel", N.METRIC_SOBEL_DIR)):
        res = {}

        def curve():
            res["curve"] = img.rd_curve(BS, BS, metric, LZ, LZ, 0)

        wall, dev = timed(ctx, curve, reps)
        factor, nbytes, sse = res["curve"]
        psnr = np.array([P.psnr_of(int(e), samples) for e in sse])
        say(f"{label}, {mname}: rd_curve {wall:.2f} ms wall, {len(factor)} points, bytes {int(nbytes[0])} .. {int(nbytes[-1])}, "
            f"PSNR {psnr[0]:.2f} .. {psnr[-1]:.2f} dB")
        split = sorted(dev.items(), key=lambda kv: -kv[1][0])
        say("  per call (device ms, launches): " + ", ".join(f"{k} {ms:.3f} ({n:g})" for k, (ms, n) in split))
        say(f"  {'target dB':>9} {'k':>12} {'payload B':>11} {'PSNR':>8} {'to_error ms':>11} {'shrink ms':>9}")
        finite = psnr[np.isfinite(psnr)]
        for q in (0.25, 0.5, 0.75):
            target = float(np.round(np.quantile(finite, q), 1))
            budget = P.sse_budget(target, samples)

            def to_error():
                pl, res["k"], res["sse"] = img.shrink_to_error(BS, BS, metric, budget, LZ, LZ, 0)
                res["bytes"] = pl.info()["bytes"]
                pl.free()

            w_err, _ = timed(ctx, to_error, reps)
            k = res["k"]
            w_plain, _ = timed(ctx, lambda: img.shrink(BS, BS, metric, k, LZ, 0).free(), reps)
            say(f"  {target:>9.1f} {P.api.format_shrinking_factor(k):>12} {res['bytes']:>11} {P.psnr_of(res['sse'], samples):>8.3f} "
                f"{w_err:>11.2f} {w_plain:>9.2f}")


ctx = N.Context(0)
say(f"GPU: {gpu_info()}  (name, power limit, SM clock, max SM clock)")
say(f"reps {REPS} (8K), {max(1, REPS // 3)} (32768^2); 64x64 blocks, Lanczos3 down and up, flags 0")

img = bench.synth_image_np(0, bench.IMG_W, bench.IMG_H)
d = ctx.image_upload(img)
frame_table(ctx, d, f"8K RGBA {bench.IMG_W}x{bench.IMG_H}", REPS)
d.free()
del img

import torch  # noqa: E402

S = 32768
frame = bench.synth_rows_device(torch, 0, S, S, 7, "cuda:0")
torch.cuda.synchronize()
src = ctx.image_wrap(frame.data_ptr(), S, S, 4, frame.stride(0))
frame_table(ctx, src, f"RGBA {S}x{S}", max(1, REPS // 3))
src.free()
say(f"GPU after the run: {gpu_info()}")

if OUT:
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")
