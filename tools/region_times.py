"""Region decode timings (pxz_payload_window / pxz_expand_region / pxz_container_crop) against the whole decode.
    python tools/region_times.py [reps] [--out FILE]

Frames: bench.py's synthetic 8K RGBA frame (64x64 blocks, Oklab-MAD k = 1, Lanczos3 both ways) and a 32768^2 RGBA frame of
the same generator, made on the device.  Device times come from the library's per-launch events (pxz_profile_*), wall
times from a host clock around the call and a stream synchronise; both are the median of `reps` repetitions after one
warm-up.  Payloads and images stay resident, so the region numbers include no PCIe transfer; the file path does."""
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
REPS = int(args[0]) if args else 20
OUT = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
BS, FD, FU = 64, 4, 4
SIZES = [(256, 256), (1024, 1024), (1920, 1080), (4096, 4096)]
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"(nvidia-smi not readable: {e})"
    return q


def median_ms(ctx, fn, reps=REPS):
    """(wall ms, {profile name: device ms per call}) medians / means over reps calls after one warm-up"""
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
    return float(np.median(walls)), {k: ms / reps for k, (ms, n) in prof.items() if n}


def region_table(ctx, pl, W, H, label, check):
    full = ctx.image_alloc(W, H, 4)
    wall, dev = median_ms(ctx, lambda: pl.expand_to_image(FU, full))
    say(f"{label}: whole pxz_expand_to_image {W}x{H}: wall {wall:.3f} ms, resample_up {dev.get('resample_up', 0) * 1e3:.1f} us")
    say(f"  {'region':>14} {'aligned':>8} {'tiles':>6} {'wall ms':>8} {'window us':>10} {'expand us':>10} {'copy us':>8} {'vs whole':>9}")
    for (w, h) in SIZES:
        if w > W or h > H:
            continue
        for aligned in (True, False):
            x = (W // 2 // BS) * BS - (w // 2 // BS) * BS
            y = (H // 2 // BS) * BS - (h // 2 // BS) * BS
            if not aligned:
                x, y = x + 37, y + 23
            x, y = max(0, min(x, W - w)), max(0, min(y, H - h))
            out = ctx.image_alloc(w, h, 4)
            rw, rdev = median_ms(ctx, lambda: pl.expand_region_to_image(FU, x, y, w, h, out))
            tiles = ((x + w - 1) // BS - x // BS + 1) * ((y + h - 1) // BS - y // BS + 1)
            say(f"  {f'{w}x{h}':>14} {'yes' if aligned else 'no':>8} {tiles:>6} {rw:>8.3f} {rdev.get('payload_window', 0) * 1e3:>10.1f} "
                f"{rdev.get('resample_up', 0) * 1e3:>10.1f} {rdev.get('region_copy', 0) * 1e3:>8.1f} {rw / wall:>8.1%}")
            if check:  # spot check: the region is the crop of the whole decode
                assert np.array_equal(out.download(), full.download()[y:y + h, x:x + w]), "region differs from the whole decode"
            out.free()
    full.free()


ctx = N.Context(0)
say(f"GPU: {gpu_info()}  (name, power limit, max SM clock)")
say(f"reps {REPS} (median wall, mean device time per call)")

# ---- 8K frame, payload resident ----------------------------------------------------------------------------------------
img = bench.synth_image_np(0, bench.IMG_W, bench.IMG_H)
d = ctx.image_upload(img)
pl8 = d.shrink(BS, BS, N.METRIC_OKLAB_MAD, 1.0, FD, 0)
region_table(ctx, pl8, bench.IMG_W, bench.IMG_H, "8K RGBA 7680x4320", True)

# fused arithmetic: do the two resample kernel families give the same pixels?
fam = {}
for kind in ("warp", "cta"):
    os.environ["PXZ_RESAMPLE_KERNELS"] = kind
    c = N.Context(0)
    del os.environ["PXZ_RESAMPLE_KERNELS"]
    c.set_fast_resample(True)
    dd = c.image_upload(img)
    p = dd.shrink(BS, BS, N.METRIC_OKLAB_MAD, 1.0, FD, 0)
    fam[kind] = p.expand(FU)
    p.free(); dd.free(); c.close()
diff = np.abs(fam["warp"].astype(np.int16) - fam["cta"]).max()
say(f"fused mode, 8K frame: warp-per-tile vs CTA-per-tile expand: {'identical' if diff == 0 else f'differ, max |diff| {diff}'} "
    f"({int((fam['warp'] != fam['cta']).sum())} bytes differ)")
pl8.free(); d.free()
del img, fam

# ---- 32768^2 frame, made on the device --------------------------------------------------------------------------------
import torch  # noqa: E402

S = 32768
frame = bench.synth_rows_device(torch, 0, S, S, 7, "cuda:0")
torch.cuda.synchronize()
src = ctx.image_wrap(frame.data_ptr(), S, S, 4, frame.stride(0))
pl = src.shrink(BS, BS, N.METRIC_OKLAB_MAD, 1.0, FD, 0)
ctx.synchronize()
src.free()
del frame
torch.cuda.empty_cache()
region_table(ctx, pl, S, S, "RGBA 32768x32768", False)

# ---- the file path on the 32768^2 file ---------------------------------------------------------------------------------
data = pl.to_container(FD, True)
pl.free()
say(f"file of the 32768^2 frame: {len(data) / 1e6:.1f} MB")
say(f"  {'region':>14} {'header+crop ms':>15} {'uploaded MB':>12} {'qoi_decode us':>14} {'expand us':>10} {'wall ms':>8}")
for (w, h) in SIZES:
    x, y = S // 2 - w // 2 + 37, S // 2 - h // 2 + 23

    def crop():
        hdr = N.container_header(data)
        c0, r0 = x // hdr["bw"], y // hdr["bh"]
        return c0, r0, N.container_crop(data, c0, r0, (x + w - 1) // BS - c0 + 1, (y + h - 1) // BS - r0 + 1)

    t_crop = []
    for _ in range(REPS):
        t = time.perf_counter()
        c0, r0, sub = crop()
        t_crop.append((time.perf_counter() - t) * 1e3)
    out = ctx.image_alloc(w, h, 4)

    def region():
        p, _ = ctx.payload_from_container(sub)
        p.expand_region_to_image(FU, x - c0 * BS, y - r0 * BS, w, h, out)
        p.free()

    rw, rdev = median_ms(ctx, region)
    rw_all, _ = median_ms(ctx, lambda: P.Pixlzr.decode_vec_region_to_image(data, P.FilterType.Lanczos3, x, y, w, h, ctx=ctx))
    say(f"  {f'{w}x{h}':>14} {np.median(t_crop):>15.3f} {len(sub) / 1e6:>12.2f} {rdev.get('qoi_decode', 0) * 1e3:>14.1f} "
        f"{rdev.get('resample_up', 0) * 1e3:>10.1f} {rw_all:>8.2f}")
    out.free()
say("  wall ms: Pixlzr.decode_vec_region_to_image end to end (header, crop, upload, decode, region, download)")

full = ctx.image_alloc(S, S, 4)


def whole():
    p, _ = ctx.payload_from_container(data)
    p.expand_to_image(FU, full)
    p.free()


w_dev, dev = median_ms(ctx, whole, reps=3)
t = time.perf_counter()
P.Pixlzr.decode_vec_to_image(data, P.FilterType.Lanczos3, ctx=ctx)
w_api = (time.perf_counter() - t) * 1e3
say(f"whole file: payload_from_container + expand_to_image {w_dev:.1f} ms wall (qoi_decode {dev.get('qoi_decode', 0):.2f} ms, "
    f"resample_up {dev.get('resample_up', 0):.2f} ms); Pixlzr.decode_vec_to_image {w_api:.0f} ms (one call, 4.3 GB download included)")
full.free()

if OUT:
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")
