"""Rate-distortion optimised encode: pxz_rdo_curve timings, and what choosing every block's size saves against one factor.
    python tools/rdo_times.py [reps] [--out FILE]

Frames: bench.py's synthetic 8K RGBA frame and a 32768^2 RGBA frame of the same generator, made on the device; 64x64
blocks, Lanczos3 down and up.  Wall times come from a host clock around the call and a stream synchronise (median of `reps`
calls after one warm-up; the 32768^2 frame runs max(1, reps // 3) calls); device times from the library's per-launch events
(pxz_profile_*), mean per call.  CUB's merge sort and scan count as one launch each.  The comparison: at four PSNR targets the
payload bytes of pxz_rdo_shrink_to_error against pxz_shrink_to_error (both metrics), and at three byte budgets the PSNR of
pxz_rdo_shrink_to_size against pxz_shrink_to_size (both metrics; its decode measured with pxz_image_error)."""
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
METRICS = (("Oklab-MAD", N.METRIC_OKLAB_MAD), ("Sobel", N.METRIC_SOBEL_DIR))
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
    res = {}

    def curve():
        res["curve"] = img.rdo_curve(BS, BS, LZ, LZ)

    wall, dev = timed(ctx, curve, reps)
    nbytes, sse = res["curve"]
    say(f"{label}: rdo_curve {wall:.2f} ms wall, {len(nbytes)} points, bytes {int(nbytes[0])} .. {int(nbytes[-1])}, "
        f"PSNR {P.psnr_of(int(sse[0]), samples):.2f} .. {P.psnr_of(int(sse[-1]), samples):.2f} dB")
    split = sorted(dev.items(), key=lambda kv: -kv[1][0])
    say("  per call (device ms, launches): " + ", ".join(f"{k} {ms:.3f} ({n:g})" for k, (ms, n) in split))
    say(f"  {'target dB':>9} {'RDO bytes':>11} {'Oklab-MAD':>11} {'Sobel':>11}   (payload bytes reaching the target)")
    for target in (30.0, 35.0, 40.0, 45.0):
        budget = P.sse_budget(target, samples)
        row = []
        pl, b, _ = img.rdo_shrink_to_error(BS, BS, budget, LZ, LZ)
        pl.free()
        row.append(b)
        for _, metric in METRICS:
            try:
                pl, _, _ = img.shrink_to_error(BS, BS, metric, budget, LZ, LZ, 0)
                row.append(pl.info()["bytes"])
                pl.free()
            except N.PixlzrError:
                row.append("unreachable")
        say(f"  {target:>9.1f} " + " ".join(f"{v:>11}" for v in row))
    say(f"  {'budget B':>11} {'RDO dB':>9} {'Oklab-MAD':>9} {'Sobel':>9}   (PSNR within the byte budget)")
    for q in (0.1, 0.25, 0.5):
        max_bytes = int(int(nbytes[0]) + q * (int(nbytes[-1]) - int(nbytes[0])))
        row = []
        pl, _, s = img.rdo_shrink_to_size(BS, BS, max_bytes, LZ, LZ)
        pl.free()
        row.append(P.psnr_of(s, samples))
        for _, metric in METRICS:
            pl, _ = img.shrink_to_size(BS, BS, metric, max_bytes, LZ, 0)
            row.append(P.psnr_of(pl.error(img, LZ)[2], samples))
            pl.free()
        say(f"  {max_bytes:>11} " + " ".join(f"{v:>9.3f}" for v in row))
    for mname, metric in METRICS:
        wall, _ = timed(ctx, lambda: img.rd_curve(BS, BS, metric, LZ, LZ, 0), reps)
        say(f"  for comparison: rd_curve {mname} {wall:.2f} ms wall")


ctx = N.Context(0)
say(f"GPU: {gpu_info()}  (name, power limit, SM clock, max SM clock)")
say(f"reps {REPS} (8K), {max(1, REPS // 3)} (32768^2); 64x64 blocks, Lanczos3 down and up")

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
