"""Rate control timings: pxz_shrink_to_size against pxz_shrink at the factor it chose.
    python tools/size_target_times.py [reps] [--out FILE]

Frames: bench.py's synthetic 8K RGBA frame and a 32768^2 RGBA frame of the same generator, made on the device; 64x64
blocks, Oklab-MAD, Lanczos3.  Budgets: fractions of the payload at k = FLT_MAX.  Wall times come from a host clock around
the call and a stream synchronise (median of `reps` calls after one warm-up); device times from the library's per-launch
events (pxz_profile_*), mean per call.  Rounds and verification passes are counted from those events: every search round
and every verification is one size_curve launch, every verification adds two guard-band recomputes (mad_exact) to the
one the final encode runs."""
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
REPS = int(args[0]) if args else 10
OUT = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
BS, FD = 64, 4
FLT_MAX = float(np.finfo(np.float32).max)
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


def timed(ctx, fn, reps=REPS):
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


def frame_table(ctx, img, label):
    full = img.shrink(BS, BS, N.METRIC_OKLAB_MAD, FLT_MAX, FD, 0)
    full_bytes = full.info()["bytes"]
    full.free()
    say(f"{label}: payload at k = FLT_MAX {full_bytes / 1e6:.1f} MB")
    say(f"  {'budget':>8} {'k':>12} {'bytes/budget':>12} {'to_size ms':>10} {'shrink ms':>9} {'overhead':>9} "
        f"{'size_curve us':>13} {'launches':>8} {'rounds':>6} {'passes':>6}")
    for frac in (0.05, 0.15, 0.3, 0.5, 0.8):
        budget = int(full_bytes * frac)
        res = {}

        def sized():
            pl, res["k"] = img.shrink_to_size(BS, BS, N.METRIC_OKLAB_MAD, budget, FD, 0)
            res["bytes"] = pl.info()["bytes"]
            pl.free()

        w_sized, dev = timed(ctx, sized)
        k = res["k"]

        def plain():
            img.shrink(BS, BS, N.METRIC_OKLAB_MAD, k, FD, 0).free()

        w_plain, _ = timed(ctx, plain)
        curve_ms, curve_n = dev.get("size_curve", (0.0, 0.0))
        passes = (dev.get("mad_exact", (0.0, 0.0))[1] - 1) / 2
        say(f"  {frac:>8.2f} {P.api.format_shrinking_factor(k):>12} {res['bytes'] / budget:>12.4f} {w_sized:>10.2f} {w_plain:>9.2f} "
            f"{w_sized - w_plain:>9.2f} {curve_ms * 1e3 / max(curve_n, 1):>13.1f} {curve_n:>8.1f} {curve_n - passes:>6.1f} {passes:>6.1f}")
    say("  overhead: to_size ms - shrink ms (wall); size_curve us: mean device time of one launch; rounds: search rounds of all "
        "passes (a pass = one search + one verification launch; a second pass runs when the first verification corrects the bracket)")


ctx = N.Context(0)
say(f"GPU: {gpu_info()}  (name, power limit, SM clock, max SM clock)")
say(f"reps {REPS}; budget as a fraction of the payload at k = FLT_MAX")

img = bench.synth_image_np(0, bench.IMG_W, bench.IMG_H)
d = ctx.image_upload(img)
frame_table(ctx, d, f"8K RGBA {bench.IMG_W}x{bench.IMG_H}")
d.free()
del img

import torch  # noqa: E402

S = 32768
frame = bench.synth_rows_device(torch, 0, S, S, 7, "cuda:0")
torch.cuda.synchronize()
src = ctx.image_wrap(frame.data_ptr(), S, S, 4, frame.stride(0))
frame_table(ctx, src, f"RGBA {S}x{S}")
src.free()
say(f"GPU after the run: {gpu_info()}")

if OUT:
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")
