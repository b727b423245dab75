"""Decode error timings: k_block_error against the stream limit, and one pxz_strategy_measure call.
    python tools/quality_times.py [reps] [--out FILE]

Frames: bench.py's synthetic 8K frame (RGBA, and its first three channels as an RGB image) and a 32768^2 RGBA frame of the
same generator made on the device; each is compared with a second image of its size (the 8K frames with their own shrink +
expand decode, the 32768^2 frame with its vertical flip).  Both images of a comparison together exceed the 126 MB L2, so
every pass streams from HBM.  32x32 blocks.  Kernel times come from the library's per-launch CUDA events (pxz_profile_*),
mean over `reps` calls after one warm-up; GB/s counts the algorithmic bytes, 2 * W * H * C read.  The strategy measure is
timed with a host clock around the call (it ends in a stream synchronise), median of `reps` calls, with the device time per
kernel from the same events.  Last, for information only: in how many of the 65 buckets a table fitted to Big-Ruscher.png
(32x32) / base.png (64x64) names the same (down, up) pair as the table of the reference author's log
(tests/golden/strategies.json); that log's criterion is not recorded, so the figure is not a check."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import pixlzr_b200 as P  # noqa: E402

N = P.native
args = [a for a in sys.argv[1:] if not a.startswith("--")]
REPS = int(args[0]) if args else 20
OUT = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
BS = 32
STREAM_LIMIT = (4.4e12, 5.1e12)  # tile-order reads of one 8K frame, profiles/r02_ubench_stream.txt
HBM = 7.7e12                     # data-sheet HBM3e bandwidth of one B200
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


def profiled(ctx, fn, reps):
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


def error_row(ctx, a, b, label):
    w, h, c = a.w, a.h, a.c
    _, dev = profiled(ctx, lambda: a.error(b, BS, BS), REPS)
    ms, n = dev["block_error"]
    us = ms * 1e3 / n
    gbs = 2.0 * w * h * c / (us * 1e-6) / 1e9
    say(f"  {label:<22} {2 * w * h * c / 1e6:>9.1f} {us:>9.1f} {gbs:>8.0f} {gbs * 1e9 / HBM * 100:>7.1f} "
        f"{gbs * 1e9 / STREAM_LIMIT[1] * 100:>5.1f}-{gbs * 1e9 / STREAM_LIMIT[0] * 100:<5.1f}")


ctx = N.Context(0)
say(f"GPU: {gpu_info()}  (name, power limit, SM clock, max SM clock)")
say(f"reps {REPS}; {BS}x{BS} blocks")
say("k_block_error (one launch per comparison; MB = algorithmic bytes 2*W*H*C)")
say(f"  {'frame':<22} {'MB':>9} {'us':>9} {'GB/s':>8} {'%7.7TB':>7} {'% of 4.4-5.1 TB/s':>17}")

img = bench.synth_image_np(0, bench.IMG_W, bench.IMG_H)
for label, x in ((f"8K RGBA {bench.IMG_W}x{bench.IMG_H}", img), (f"8K RGB {bench.IMG_W}x{bench.IMG_H}", np.ascontiguousarray(img[..., :3]))):
    a = ctx.image_upload(x)
    pl = a.shrink(BS, BS, N.METRIC_OKLAB_MAD, 1.0, int(P.FilterType.Lanczos3))
    b = ctx.image_alloc(a.w, a.h, a.c)
    pl.expand_to_image(int(P.FilterType.Lanczos3), b)
    pl.free()
    error_row(ctx, a, b, label)
    a.free(), b.free()

import torch  # noqa: E402

S = 32768
frame = bench.synth_rows_device(torch, 0, S, S, 7, "cuda:0")
other = frame.flip(0).contiguous()
torch.cuda.synchronize()
fa = ctx.image_wrap(frame.data_ptr(), S, S, 4, frame.stride(0))
fb = ctx.image_wrap(other.data_ptr(), S, S, 4, other.stride(0))
error_row(ctx, fa, fb, f"RGBA {S}x{S}")
fa.free(), fb.free()
del frame, other
torch.cuda.empty_cache()

say()
say(f"pxz_strategy_measure, 8K RGBA, {BS}x{BS}, Oklab-MAD, factor 1: 5 shrinks + 25 expands + 25 error / bucket passes")
a = ctx.image_upload(img)
wall, dev = profiled(ctx, lambda: a.strategy_measure(BS, BS, N.METRIC_OKLAB_MAD, 1.0, 0), max(3, REPS // 4))
say(f"  wall {wall:.2f} ms per call (median); device ms per call by kernel (launches per call):")
say("  " + ", ".join(f"{k} {ms:.3f} ({n:g})" for k, (ms, n) in sorted(dev.items(), key=lambda kv: -kv[1][0])))
say(f"  sum of kernel times {sum(ms for ms, _ in dev.values()):.2f} ms")
a.free()

say()
say("table fitted per bucket (Strategy.fit) against the author's logged table (tests/golden/strategies.json), for information only:")
with open(os.path.join(ROOT, "tests", "golden", "strategies.json")) as f:
    # the buckets the author measured; the log goes beyond v = 1, and all of those are bucket 64's (Nearest, Nearest)
    logged = {min(int(b), 64): d * 5 + u for b, (d, u) in json.load(f)["per_bucket"].items()}
from PIL import Image  # noqa: E402

ims = [(np.array(Image.open(os.path.join(ROOT, "tests", "golden", n))), bs) for n, bs in (("Big-Ruscher.png", 32), ("base.png", 64))]
for factor in (0.2, 1.0):
    sse = np.zeros((N.STRATEGY_BUCKETS, N.FILTER_PAIRS), np.uint64)
    blocks = np.zeros(N.STRATEGY_BUCKETS, np.uint32)
    for im, bs in ims:
        _, rep = P.Strategy.fit([im], bs, bs, factor, ctx=ctx)
        sse += rep.sse
        blocks += rep.blocks
    fit = P.Strategy(*N.strategy_choose(sse, blocks))
    rep = P.StrategyReport(sse, blocks)
    pairs = fit.down.astype(np.int64) * 5 + fit.up
    both = [b for b in sorted(logged) if blocks[b] > 0]  # measured by the author and holding blocks here
    same = sum(int(pairs[b] == logged[b]) for b in both)
    say(f"  factor {factor}: {int((blocks > 0).sum())} buckets hold blocks, {len(both)} of them measured in the log; same pair as the log "
        f"in {same} of those {len(both)}; summed squared error fitted {rep.total(fit)} / logged table (by_level) "
        f"{rep.total(P.Strategy.by_level())} / uniform Lanczos3 {rep.total(P.Strategy.uniform(4, 4))}")
say(f"GPU after the run: {gpu_info()}")

if OUT:
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")
