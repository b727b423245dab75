#!/usr/bin/env python3
"""bench.py — encode+decode megapixels/s of the pixlzr hot path on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Headline workload (BASELINE.json configs[2], "C3"): synthetic 7680x4320 RGBA8 frames, 64x64 blocks, metric
Oklab-MAD with k = 1, Lanczos3 down / Lanczos3 up (the reference CLI's defaults, src/bin/main.rs:19,27-36).
One step = encode (analyse -> plan -> shrink into the packed payload) + decode (expand + paste) of `--batch`
frames per rank (`--distinct` different ones, taken in turn: 531 MB of input, larger than L2); frames are
independent, so ranks share nothing (weak scaling) and no collective sits on the data path.  `value` is timed
with CUDA events on the launching stream with every input already resident in HBM; `e2e` runs the same work
through the C ABI with pinned HOST buffers, host<->device copies inside the timed region.

The same line carries the two sharded configurations of BASELINE.json, measured on the same N ranks:
  "sharded": C4, one 65536 x 65536 frame (generated on the device) cut into block-row shards, once with the
             global-normalisation extension (the library's NCCL min/max all-reduce is the only exchange) and once
             in the default mode; a checksum of descriptors and payload that must not depend on N;
  "batch":   C5, 4096 frames of 1920x1080 dealt round-robin, through the batch entry points of the C ABI
             (pxz_shrink_batch / pxz_expand_batch: one launch per stage over a stack of frames);
and, at N >= 2, "nccl_parity": the sharded result of a small frame equals the single-GPU result, including ranks
without rows and a rank that fails before the exchange.  Prints ONE JSON line on rank 0.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step gave its caller for the frames whose decodes
are still in the output buffers (one per stream) as DIR/<name>.npy (see dump_outputs).  The inputs depend on the
arguments only, so two builds run with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "encode+decode megapixels/sec"
UNIT = "MP/s"
BS = 64
FILTER_DOWN = 4  # Lanczos3
FILTER_UP = 4
FACTOR = 1.0
IMG_W, IMG_H = 7680, 4320
CPU_SAMPLE_ROWS = 1088  # 17 block rows of the 8K frame = 8.36 MP: the bounded sample of the in-run CPU baseline


# --------------------------------------------------------------------------------------------------
# synthetic input (BASELINE.md section 3): slow colour ramps + per-64x64-tile uniform noise whose amplitude
# is picked from {0,1,2,4,8,16,32,64} by a tile hash, so that every level 2^0 .. 2^-6 occurs
# --------------------------------------------------------------------------------------------------
def synth_image_np(seed: int, w: int, h: int) -> np.ndarray:
    rng = np.random.default_rng(0x5049584C5A52 ^ seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.stack([128 + 96 * np.sin(xx / 9000.0 + seed), 128 + 96 * np.cos(yy / 7000.0 + 0.3 * seed),
                     128 + 64 * np.sin((xx + yy) / 11000.0)], -1)
    ty, tx = np.mgrid[0:(h + 63) // 64, 0:(w + 63) // 64].astype(np.uint64)
    hsh = (tx * np.uint64(73856093)) ^ (ty * np.uint64(19349663)) ^ np.uint64((seed * 83492791) & 0xFFFFFFFF)
    amp = np.array([0, 1, 2, 4, 8, 16, 32, 64], np.float32)[(hsh >> np.uint64(3)) % np.uint64(8)]
    amp = np.kron(amp, np.ones((64, 64), np.float32))[:h, :w]
    img = base + (rng.random((h, w, 3), dtype=np.float32) - 0.5) * 2 * amp[..., None]
    img = np.clip(np.rint(img), 0, 255).astype(np.uint8)
    return np.ascontiguousarray(np.concatenate([img, np.full((h, w, 1), 255, np.uint8)], -1))


class DeviceSynth:
    """Frames generated on the device: smooth base + per-64x64-tile noise whose amplitude is a hash of the tile, alpha 255.
    The generator is seeded per 64-row band of the FRAME, so the pixels depend neither on the sharding nor on its layout
    (contiguous runs or interleaved block rows).  Used for the frames that are too large to cross PCIe (C4) or too many (C5)."""

    BAND = 64

    def __init__(self, torch, width, seed, device):
        self.torch, self.width, self.seed, self.device = torch, width, seed, device
        self.xx = torch.arange(width, device=device, dtype=torch.float32)
        self.tx = (torch.arange(width, device=device) // 64).to(torch.int64)
        self.amps = torch.tensor([0, 1, 2, 4, 8, 16, 32, 64], device=device, dtype=torch.float32)

    def band(self, g0, out):
        """rows [g0, g0 + out.shape[0]) of the frame (g0 a multiple of 64, at most 64 rows) into out[:, :, 0:3]"""
        torch, seed, n = self.torch, self.seed, self.BAND
        yy = torch.arange(g0, g0 + n, device=self.device, dtype=torch.float32)[:, None]
        ty = (torch.arange(g0, g0 + n, device=self.device) // 64).to(torch.int64)[:, None]
        h = (ty * 73856093 + self.tx[None, :] * 19349663 + seed * 83492791) & 0x7FFFFFFF
        amp = self.amps[(h >> 7) % 8]
        g = torch.Generator(device=self.device)
        g.manual_seed(seed * 1000003 + g0)
        xx = self.xx
        for ch, base in enumerate((128 + 96 * torch.sin(xx[None, :] / 9700.0 + seed), 128 + 96 * torch.cos(yy / 13100.0),
                                   128 + 64 * torch.sin((xx[None, :] + yy) / 6100.0))):
            noise = (torch.rand((n, self.width), device=self.device, generator=g) - 0.5) * 2 * amp
            full = torch.clamp(torch.round(base + noise), 0, 255).to(torch.uint8)
            out[:, :, ch] = full[:out.shape[0]]


def synth_rows_device(torch, y0, y1, width, seed, device):
    """uint8 [y1-y0, width, 4] on the device: rows [y0, y1) of the synthetic frame (y0 a multiple of 64)."""
    out = torch.empty((y1 - y0, width, 4), dtype=torch.uint8, device=device)
    out[..., 3] = 255
    syn = DeviceSynth(torch, width, seed, device)
    for g0 in range(y0, y1, DeviceSynth.BAND):
        syn.band(g0, out[g0 - y0:min(y1, g0 + DeviceSynth.BAND) - y0])
    return out


def synth_block_rows_device(torch, rows_idx, height, width, seed, device):
    """The same frame's block rows `rows_idx` (64 px each) stacked: a rank's local image in the interleaved layout."""
    hs = [min(height, (g + 1) * 64) - g * 64 for g in rows_idx]
    out = torch.empty((sum(hs), width, 4), dtype=torch.uint8, device=device)
    out[..., 3] = 255
    syn = DeviceSynth(torch, width, seed, device)
    y = 0
    for g, n in zip(rows_idx, hs):
        syn.band(g * 64, out[y:y + n])
        y += n
    return out


class ClockSampler:
    """SM clock and throttle reasons of one GPU while the timed region runs: NVML polled in-process from one thread
    (no child processes next to the timed region); falls back to one nvidia-smi query before and after."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index: int, period_s: float = 0.01):
        self.gpu, self.period, self.samples, self.stop_flag = gpu_index, period_s, [], threading.Event()
        self.nv = self.handle = self.thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.handle = pynvml, pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else 0x8,
                "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        while not self.stop_flag.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.samples.append((time.time(), float(mhz), [n for n, b in bits.items() if r & b]))
            except Exception:
                pass
            self.stop_flag.wait(self.period)

    def _smi_once(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            o = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                               capture_output=True, text=True, timeout=10).stdout.strip().split(",")
            self.samples.append((time.time(), float(o[0]), [n for n, v in zip(self.NAMES, o[2:6]) if v.strip().lower().startswith("active")]))
            self.smax = float(o[1])
        except Exception:
            pass

    def start(self):
        if self.nv is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        else:
            self._smi_once()

    def stop(self, t0: float, t1: float) -> dict:
        smax = None
        if self.nv is not None:
            self.stop_flag.set()
            self.thread.join(timeout=1.0)
            try:
                smax = float(self.nv.nvmlDeviceGetMaxClockInfo(self.handle, self.nv.NVML_CLOCK_SM))
            except Exception:
                pass
        else:
            self._smi_once()
            smax = getattr(self, "smax", None)
        rows = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples
        reasons = sorted({r for _, _, rs in rows for r in rs})
        return {"sm_mhz": float(np.median([m for _, m, _ in rows])) if rows else None, "sm_max_mhz": smax, "reasons": reasons,
                "samples": len(rows), "source": "NVML, in-process, every 10 ms inside the timed region" if self.nv is not None else
                "nvidia-smi before and after the timed region (NVML unavailable)"}


# --------------------------------------------------------------------------------------------------
# CPU legs (oracle = C++ port of the reference; the Rust reference itself cannot be built here)
# --------------------------------------------------------------------------------------------------
def cpu_encode_decode(O, sample: np.ndarray, threads: int):
    t0 = time.perf_counter()
    s = O.shrink(sample, BS, BS, O.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, nthreads=threads)
    out = O.expand(s, FILTER_UP, nthreads=threads)
    return time.perf_counter() - t0, s, out


def cpu_baseline(sample: np.ndarray):
    import oracle as O

    cores = os.cpu_count() or 1
    mp = sample.shape[0] * sample.shape[1] / 1e6
    cpu_encode_decode(O, sample, cores)  # warm-up (thread pool, page faults)
    runs = [cpu_encode_decode(O, sample, cores) for _ in range(5)]
    best_all = min(r[0] for r in runs)
    best_one = min(cpu_encode_decode(O, sample, 1)[0] for _ in range(2))
    info = {"value": mp / best_all, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"top {sample.shape[0]} rows ({mp:.2f} MP) of frame 0 of the same workload, best of 5",
            "one_thread_value": mp / best_one,
            "note": "shrink* is a serial loop in the reference (pixlzr.rs:163-184); the all-core figure is charitable"}
    return info, runs[-1][1], runs[-1][2]


def workload_config(args) -> dict:
    return {
        "workload": "C3 synthetic 7680x4320 RGBA8 (alpha 255), 64x64 blocks, Oklab-MAD k=1, Lanczos3 down / Lanczos3 up, "
                    "encode (analyse+plan+shrink) + decode (expand+paste)",
        "width": IMG_W, "height": IMG_H, "channels": 4, "block": BS, "metric": "oklab_mad", "factor": FACTOR,
        "filter_down": "Lanczos3", "filter_up": "Lanczos3", "images_per_step_per_gpu": args.batch,
        "distinct_images_per_gpu": min(args.distinct, args.batch),
        "sharding": "independent images per rank, no data-path collective",
        "cache": "inputs larger than L2 (the distinct frames of a rank are 531 MB and are taken in turn)",
        "resize_semantics": "image_rs (the branch pinned by the reference's fixtures)",
    }


def run_reference(args, rank: int):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the Rust crate cannot be built in
    this image: no cargo/rustc) on all host cores, SAME frames, same images per step."""
    if rank != 0:
        return
    import oracle as O

    cores = os.cpu_count() or 1
    distinct = min(args.distinct, args.batch)
    frames = [synth_image_np(i, IMG_W, IMG_H) for i in range(distinct)]
    mp_step = args.batch * IMG_W * IMG_H / 1e6

    def step():
        for i in range(args.batch):
            cpu_encode_decode(O, frames[i % distinct], cores)
    for _ in range(min(args.warmup, 1)):  # one full step warms the thread pool and the page cache: more would only cost minutes
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    val = mp_step * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"each step = the same {args.batch} full 8K frames ({mp_step:.0f} MP) as the B200 arm; "
                                   f"warm-up capped at one step"},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# B200 arm: helpers
# --------------------------------------------------------------------------------------------------
def timed_region(torch, dist, world, device, fn, reps):
    """max over ranks of the mean device-side time of fn (barrier + synchronize on both sides, CUDA events on the
    current stream; fn must leave every stream it uses joined into the current one)."""
    fn()
    torch.cuda.synchronize(device)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize(device)
    ms = torch.tensor([e0.elapsed_time(e1) / reps], device=device, dtype=torch.float64)
    mine = float(ms.item())
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), mine


DUMP_BYTES = 64 << 20  # --dump-outputs writes at most this much in all
DUMP_SEED = 0x44554D50


def dump_outputs(out_dir: str, decoded: list, descs: list, payloads: list) -> int:
    """Writes the encode + decode results of F frames as out_dir/<name>.npy and returns the bytes written:
      block_offset (float64), block_value / block_width / block_height (float32)   [F, blocks]  every descriptor
      payload_bytes (float64) [F]                                                   payload size of each frame
      payload_sample (float32) [F, Q]       Q payload bytes at seeded positions (the same ones for equal sizes)
      decoded_sample (float32) [F, P, C]    P decoded pixels at seeded positions (the same ones in every frame)
    An 8K RGBA frame is 133 MB, so P and Q are chosen to keep the files within DUMP_BYTES."""
    n = len(decoded)
    h, w, c = decoded[0].shape
    npx = h * w
    n_pix = min(npx, (DUMP_BYTES // 2) // (4 * c * n))
    n_pay = min([p.size for p in payloads] + [(DUMP_BYTES // 4) // (4 * n)])
    pix_idx = np.sort(np.random.default_rng(DUMP_SEED).choice(npx, n_pix, replace=False))
    arrays = {
        "block_offset": np.stack([d["offset"] for d in descs]).astype(np.float64),
        "block_value": np.stack([d["value"] for d in descs]).astype(np.float32),
        "block_width": np.stack([d["w"] for d in descs]).astype(np.float32),
        "block_height": np.stack([d["h"] for d in descs]).astype(np.float32),
        "payload_bytes": np.array([p.size for p in payloads], np.float64),
        "payload_sample": np.stack([p[np.sort(np.random.default_rng(DUMP_SEED).choice(p.size, n_pay, replace=False))]
                                    for p in payloads]).astype(np.float32),
        "decoded_sample": np.stack([img.reshape(npx, c)[pix_idx] for img in decoded]).astype(np.float32),
    }
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes of outputs exceed {DUMP_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return total


def run_sharded_c4(torch, dist, N, S, args, rank, world, local_rank, device):
    """C4: one side x side frame in block-row shards, contiguous runs and interleaved rows; global normalisation = the only
    exchange."""
    side = args.c4_side
    ctx = N.Context(local_rank, cuda_stream=torch.cuda.current_stream(device).cuda_stream)
    if world > 1:
        S.init_comm(ctx, dist, rank, world, device=device)

    def measure(src, flags):
        """encode+decode of this rank's rows `src` [rows, side, 4]: whole-job MP/s, per-rank ms, checksum over all ranks"""
        dst = torch.empty_like(src)
        img = ctx.image_wrap(src.data_ptr(), side, src.shape[0], 4, side * 4)
        out = ctx.image_wrap(dst.data_ptr(), side, src.shape[0], 4, side * 4)

        def step():
            pl = img.shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, flags)
            pl.expand_to_image(FILTER_UP, out)
            pl.free()
        ms, mine = timed_region(torch, dist, world, device, step, args.extra_reps)
        pl = img.shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, flags)
        descs, px = pl.download()
        pl.free()
        chk = torch.tensor([int(descs["w"].astype(np.uint64).sum() * 65537 + descs["h"].astype(np.uint64).sum()),
                            int(px.astype(np.uint64).sum()), int(px.size)], device=device, dtype=torch.int64)
        per_rank = torch.tensor([mine], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(chk)
            g = [torch.zeros_like(per_rank) for _ in range(world)]
            dist.all_gather(g, per_rank)
            per_rank_ms = [round(float(t.item()), 3) for t in g]
        else:
            per_rank_ms = [round(mine, 3)]
        return {"MPps": round(side * side / (ms / 1e3) / 1e6, 1), "ms": round(ms, 3), "ms_per_rank": per_rank_ms,
                "payload_fraction": round(int(chk[2]) / (side * side * 4), 4), "checksum": [int(chk[0]), int(chk[1])]}

    modes = (("normalise_global", N.FLAG_NORMALISE_GLOBAL), ("default", 0))
    res = {}
    y0, y1 = S.shard_pixel_rows(side, BS, world, rank)
    src = synth_rows_device(torch, y0, y1, side, 7, device)
    for name, flags in modes:
        res[name] = measure(src, flags)
    del src
    torch.cuda.empty_cache()
    # both modes again with INTERLEAVED block rows (row g of the frame on rank g mod N, sharding.cyclic_block_rows):
    # the cost of a block row follows the frame's content, which changes slowly down the frame, so contiguous runs are
    # uneven (two of eight ranks carry 40 % more work above) while every N-th row gives each rank the same level mix
    src = synth_block_rows_device(torch, S.cyclic_block_rows(-(-side // BS), world, rank), side, side, 7, device)
    for name, flags in modes:
        r = measure(src, flags)
        r["same_result_as_contiguous"] = r["checksum"] == res[name]["checksum"]
        res[name + "_interleaved"] = r
    res["note"] = ("normalise_global = the extension of BASELINE config 4: v' = (v - min) / (max - min) over the whole frame, one NCCL "
                   "min all-reduce of {min, -max} per shrink (the only exchange), min and max in reference order; checksum = sum over ranks of descriptor dims and "
                   "payload bytes: it must be the same at every N and in both layouts; *_interleaved = block row g of the frame on rank g mod N")
    res["config"] = f"C4 synthetic {side}x{side} RGBA8 generated on the device, 64x64 blocks, block-row shards (contiguous runs; *_interleaved: every N-th row), Oklab-MAD k=1, Lanczos3 / Lanczos3, encode+decode, device-resident"
    res["blocks"] = (side // BS) ** 2
    del src
    torch.cuda.empty_cache()
    return res


def run_batch_c5(torch, dist, N, S, args, rank, world, local_rank, device):
    """C5: args.c5_images frames of 1920x1080 dealt round-robin; every rank runs its share in stacks of args.c5_stack frames
    through the batch entry points."""
    w, h = 1920, 1080
    mine = S.round_robin(args.c5_images, world, rank)
    stack = max(1, min(args.c5_stack, len(mine)))
    n_stacks = -(-len(mine) // stack)
    distinct_stacks = min(n_stacks, 2)  # two different stacks of `stack` different frames (2 x 530 MB at 64), taken in turn
    stream0 = torch.cuda.current_stream(device)
    streams = [stream0] + [torch.cuda.Stream(device=device) for _ in range(max(0, min(args.streams, n_stacks) - 1))]
    ctxs = [N.Context(local_rank, cuda_stream=s.cuda_stream) for s in streams]
    srcs = []
    for k in range(distinct_stacks):
        t = torch.empty((stack, h, w, 4), dtype=torch.uint8, device=device)
        for i in range(stack):
            t[i] = synth_rows_device(torch, 0, h, w, 100 + mine[(k * stack + i) % len(mine)], device)
        srcs.append(t)
    outs = [torch.empty((stack, h, w, 4), dtype=torch.uint8, device=device) for _ in ctxs]
    imgs = [[c.image_wrap_batch(t.data_ptr(), w, h, 4, w * 4, stack) for t in srcs] for c in ctxs]
    wouts = [c.image_wrap_batch(o.data_ptr(), w, h, 4, w * 4, stack) for c, o in zip(ctxs, outs)]

    def step():
        ev = torch.cuda.Event()
        ev.record(stream0)
        for s in streams[1:]:
            s.wait_event(ev)
        for n in range(n_stacks):
            k = n % len(ctxs)
            pl = imgs[k][n % distinct_stacks].shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
            pl.expand_to_image(FILTER_UP, wouts[k])
            pl.free()
        for s in streams[1:]:
            e = torch.cuda.Event()
            e.record(s)
            stream0.wait_event(e)
    ms, me = timed_region(torch, dist, world, device, step, args.extra_reps)
    done = n_stacks * stack * world  # frames actually processed (the last stack of a rank is run full)
    res = {"MPps": round(done * w * h / (ms / 1e3) / 1e6, 1), "images_per_s": round(done / (ms / 1e3)), "ms_per_pass": round(ms, 3),
           "images": done, "images_per_stack": stack, "streams_per_gpu": len(streams),
           "config": f"C5 batch of {args.c5_images} synthetic 1920x1080 RGBA8 frames round-robin over the ranks, 64x64 blocks, Oklab-MAD k=1, "
                     f"Lanczos3 / Lanczos3, encode+decode, device-resident, pxz_shrink_batch / pxz_expand_batch on stacks of {stack} frames"}
    # the same frames one call per frame (what round 1 measured): shows what the batch entry points buy
    single = [ctxs[0].image_wrap(srcs[0][i].data_ptr(), w, h, 4, w * 4) for i in range(min(stack, 16))]
    wo = ctxs[0].image_wrap(outs[0][0].data_ptr(), w, h, 4, w * 4)

    def step1():
        for im in single:
            pl = im.shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
            pl.expand_to_image(FILTER_UP, wo)
            pl.free()
    ms1, _ = timed_region(torch, dist, world, device, step1, args.extra_reps)
    res["one_call_per_image_MPps"] = round(len(single) * world * w * h / (ms1 / 1e3) / 1e6, 1)
    del srcs, outs
    torch.cuda.empty_cache()
    return res


def run_nccl_parity(torch, dist, N, S, O_or_none, rank, world, local_rank, device):
    """N >= 2: the sharded encode of a small frame (global normalisation through the library's NCCL exchange) equals the
    single-GPU encode of the whole frame; ranks without rows join the exchange; a rank that fails before the exchange does
    not leave the others waiting."""
    res = {}
    ctx = N.Context(local_rank, cuda_stream=torch.cuda.current_stream(device).cuda_stream)
    S.init_comm(ctx, dist, rank, world, device=device)
    for name, (w, h) in (("rows_ge_ranks", (328, 64 * 2 * world + 24)), ("fewer_rows_than_ranks", (328, 64 * max(1, world // 2)))):
        img = synth_image_np(900 + h, w, h)
        y0, y1 = S.shard_pixel_rows(h, BS, world, rank)
        if y1 > y0:
            d = ctx.image_upload(np.ascontiguousarray(img[y0:y1]))
            pl = d.shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, N.FLAG_NORMALISE_GLOBAL)
            descs, px = pl.download()
            pl.free(); d.free()
            mine = [int(descs["w"].astype(np.uint64).sum() * 65537 + descs["h"].astype(np.uint64).sum()), int(px.astype(np.uint64).sum()), int(px.size)]
        else:
            ctx.comm_join_empty()
            mine = [0, 0, 0]
        chk = torch.tensor(mine, device=device, dtype=torch.int64)
        dist.all_reduce(chk)
        ok = None
        if rank == 0:
            solo = N.Context(local_rank)
            d = solo.image_upload(img)
            pl = d.shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, N.FLAG_NORMALISE_GLOBAL)
            descs, px = pl.download()
            pl.free(); d.free()
            want = [int(descs["w"].astype(np.uint64).sum() * 65537 + descs["h"].astype(np.uint64).sum()), int(px.astype(np.uint64).sum()), int(px.size)]
            ok = want == [int(v) for v in chk]
        res[name] = ok
    # a rank-local failure before the exchange: the last rank's shard ends in a 1-row block, which the Sobel metric
    # refuses (the reference panics there) — every rank must come back, the healthy ones with PXZ_E_NCCL
    h = 64 * world + 1
    img = synth_image_np(77, 328, h)
    y0, y1 = S.shard_pixel_rows(h, BS, world, rank)
    status = "ok"
    try:
        d = ctx.image_upload(np.ascontiguousarray(img[y0:y1]))
        pl = d.shrink(BS, BS, N.METRIC_SOBEL_DIR, 4.0, FILTER_DOWN, N.FLAG_NORMALISE_GLOBAL)
        pl.free(); d.free()
    except N.PixlzrError as e:
        status = N.STATUS_NAMES.get(e.status, str(e.status))
    flags = torch.tensor([1 if status != "ok" else 0], device=device, dtype=torch.int64)
    dist.all_reduce(flags)
    if rank == 0:
        res["failing_rank_does_not_hang"] = int(flags.item()) == world  # every rank returned, each with an error
    return res


# --------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------
def _parse_cpulist(text: str) -> set:
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        a, _, b = part.partition("-")
        cpus.update(range(int(a), int(b or a) + 1))
    return cpus


def bind_to_gpu_numa_node(torch, local_rank: int) -> dict:
    """Run this rank's host threads on the CPUs of the NUMA node its GPU hangs off, BEFORE any pinned buffer exists:
    pinned pages are placed where the allocating thread runs, and a DMA that crosses the socket interconnect gets a
    fraction of the PCIe rate when all ranks copy at once.  A no-op (reported) when sysfs exposes no node for the GPU."""
    info = {"bound": False}
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        info["gpu_pci"] = bdf
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
        info["nodes_online"] = len(nodes)
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read().strip())
        info["node"] = node
        if node < 0 or len(nodes) < 2:
            return info
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = _parse_cpulist(f.read()) & os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            info["bound"], info["cpus"] = True, len(cpus)
    except Exception as e:  # no sysfs entry, no permission: keep the default placement
        info["error"] = repr(e)
    return info


def run_b200(args, rank: int, world: int, local_rank: int):
    import torch
    import torch.distributed as dist

    import pixlzr_b200 as P

    N, S = P.native, P.sharding
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    host_numa = bind_to_gpu_numa_node(torch, local_rank) if args.numa_bind else {"bound": False, "off": True}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(device=dev)
    batch, distinct = args.batch, min(args.distinct, args.batch)
    t_start = time.time()

    with torch.cuda.stream(stream):
        ctx = N.Context(local_rank, cuda_stream=stream.cuda_stream)
        # inputs: host (pinned) for the e2e leg, device-resident copies for the kernel leg
        # every rank gets the SAME frames (seeds 0 .. distinct-1): weak scaling means the same work per rank, and the work of a
        # frame depends on its content (the level mix); round 1 seeded by rank and two of eight ranks drew heavier frames
        host_imgs = [torch.from_numpy(synth_image_np(i, IMG_W, IMG_H)).pin_memory() for i in range(distinct)]
        dev_imgs = [t.to(dev, non_blocking=True) for t in host_imgs]
        stream.synchronize()
        # device-resident leg: `--streams` contexts (one CUDA stream each) take the frames of a step in turn, so the
        # latency-bound kernels of one frame (guard-band recompute, plan) overlap the throughput kernels of another
        n_streams = max(1, min(args.streams, batch))
        streams = [stream] + [torch.cuda.Stream(device=dev) for _ in range(n_streams - 1)]
        ctxs = [ctx] + [N.Context(local_rank, cuda_stream=st.cuda_stream) for st in streams[1:]]
        outs = [torch.empty((IMG_H, IMG_W, 4), dtype=torch.uint8, device=dev) for _ in range(n_streams)]
        wrapped = [[c.image_wrap(t.data_ptr(), IMG_W, IMG_H, 4, IMG_W * 4) for t in dev_imgs] for c in ctxs]
        wrapped_out = [ctxs[k].image_wrap(outs[k].data_ptr(), IMG_W, IMG_H, 4, IMG_W * 4) for k in range(n_streams)]

        def step_device():
            for i in range(batch):
                k = i % n_streams
                pl = wrapped[k][i % distinct].shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
                pl.expand_to_image(FILTER_UP, wrapped_out[k])
                pl.free()

        # payload sizes (for the algorithmic-byte counts), untimed
        payload_bytes, nblocks = [], 0
        for im in wrapped[0]:
            pl = im.shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
            info = pl.info()
            payload_bytes.append(info["bytes"])
            nblocks = info["cols"] * info["rows"]
            pl.free()

        for _ in range(args.warmup):
            step_device()
        if args.warmup == 0 and args.issue == "graph":
            step_device()  # every context needs its cached payload buffers and tables before a capture (no allocation, no
            #                table upload inside it)
        torch.cuda.synchronize()

        # The K timed steps are captured once into a CUDA graph (fork: every stream waits for the launching one; the K x
        # `batch` encode+decode calls through the C ABI, exactly as issued directly; join) and the timed region replays
        # it, so that the host is out of the measurement: at N = 8 eight Python issue loops share the box's 32 vCPUs and
        # two or three ranks came out 5-10 % slower with identical kernels.  `--issue direct` keeps the plain loop; a
        # capture the driver refuses falls back to it (config.issue says which ran).
        graph, issue_mode, captured_launches, graph_note = None, "direct", 0, None
        if args.issue == "graph":
            try:
                l0 = sum(c.launch_count() for c in ctxs)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=stream, capture_error_mode="relaxed"):
                    fork = torch.cuda.Event()
                    fork.record(stream)
                    for st in streams[1:]:
                        st.wait_event(fork)
                    for _ in range(args.steps):
                        step_device()
                    for st in streams[1:]:
                        e = torch.cuda.Event()
                        e.record(st)
                        stream.wait_event(e)
                captured_launches = sum(c.launch_count() for c in ctxs) - l0
                graph.replay()           # one untimed replay: uploads the executable graph
                torch.cuda.synchronize()
                issue_mode = "graph"
            except Exception as exc:     # noqa: BLE001 - any capture problem: measure with the plain loop
                graph, graph_note = None, f"graph capture failed ({type(exc).__name__}: {str(exc)[:160]}); direct issue"
                try:
                    torch.cuda.synchronize()
                except Exception:        # noqa: BLE001
                    pass
                for _ in range(2):
                    step_device()
                torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        sampler = ClockSampler(local_rank if "CUDA_VISIBLE_DEVICES" not in os.environ else
                               int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank]))
        sampler.start()
        launches0 = sum(c.launch_count() for c in ctxs)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_wall0 = time.time()
        if graph is not None:
            ev0.record(stream)
            graph.replay()
            t_launched = time.time()
            ev1.record(stream)
        else:
            ev0.record(stream)               # the timed region starts on the launching stream ...
            for st in streams[1:]:
                st.wait_event(ev0)           # ... and every other stream starts after it
            for _ in range(args.steps):
                step_device()
            t_launched = time.time()         # host time to issue the K steps (launch-bound when close to the device time)
            for st in streams[1:]:
                e = torch.cuda.Event()
                e.record(st)
                stream.wait_event(e)         # the launching stream joins all the others before the end event
            ev1.record(stream)
        stream.synchronize()
        torch.cuda.synchronize()
        t_wall1 = time.time()
        if world > 1:
            dist.barrier()
        elapsed_ms = ev0.elapsed_time(ev1)
        launches = captured_launches if graph is not None else sum(c.launch_count() for c in ctxs) - launches0
        clocks = sampler.stop(t_wall0, t_wall1)

        # ---- --dump-outputs: the last timed step's results, before the passes below overwrite the output buffers --------
        if args.dump_outputs and rank == 0:
            decoded, descs_k, payloads = [], [], []
            for k in range(n_streams):
                i = k + (batch - 1 - k) // n_streams * n_streams  # the step's last frame on stream k: its decode is in outs[k]
                got = outs[k].cpu().numpy()
                # the step freed its payloads: encode the same frame again (the encode is deterministic) and require it to
                # decode to what the timed step decoded
                pl = wrapped[0][i % distinct].shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
                descs, px = pl.download()
                again = pl.expand(FILTER_UP)
                pl.free()
                if not np.array_equal(again, got):
                    raise RuntimeError(f"--dump-outputs: frame {i} encoded again does not decode to the timed step's result")
                decoded.append(got)
                descs_k.append(descs)
                payloads.append(px)
            dump_outputs(args.dump_outputs, decoded, descs_k, payloads)
            del decoded, descs_k, payloads

        # per-kernel durations without cross-stream overlap: the same frames on the launching stream only, CUDA events
        # around every launch (pxz_profile_*).  This pass is what the roofline of the dominant kernel is computed from.
        solo_steps = max(2, min(args.steps, 6))
        ctx.profile_enable(True)
        ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev2.record(stream)
        for _ in range(solo_steps):
            for i in range(batch):
                pl = wrapped[0][i % distinct].shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
                pl.expand_to_image(FILTER_UP, wrapped_out[0])
                pl.free()
        ev3.record(stream)
        stream.synchronize()
        solo_ms = ev2.elapsed_time(ev3)
        prof = ctx.profile_read()
        ctx.profile_enable(False)
        # the same single-stream pass without the per-launch events (they cost a few microseconds per kernel)
        ev4, ev5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev4.record(stream)
        for _ in range(solo_steps):
            for i in range(batch):
                pl = wrapped[0][i % distinct].shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
                pl.expand_to_image(FILTER_UP, wrapped_out[0])
                pl.free()
        ev5.record(stream)
        stream.synchronize()
        solo_plain_ms = ev4.elapsed_time(ev5)

        # ---- in-run parity on the timed workload: frame 0, top CPU_SAMPLE_ROWS rows, against the oracle ----------------
        parity = None
        cpu = None
        if rank == 0:
            sample = np.ascontiguousarray(host_imgs[0].numpy()[:CPU_SAMPLE_ROWS])
            cpu, ref_s, ref_out = cpu_baseline(sample)
            pl = wrapped[0][0].shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
            descs, px = pl.download()
            pl.expand_to_image(FILTER_UP, wrapped_out[0])
            stream.synchronize()
            got = outs[0][:CPU_SAMPLE_ROWS].cpu().numpy()
            pl.free()
            nb = len(ref_s.descs)
            dims_ok = bool(np.array_equal(descs["w"][:nb], ref_s.descs["w"]) and np.array_equal(descs["h"][:nb], ref_s.descs["h"]) and
                           np.array_equal(descs["offset"][:nb], ref_s.descs["offset"]))
            payload_ok = bool(np.array_equal(px[:ref_s.payload.size], ref_s.payload))
            diff = np.abs(got.astype(np.int16) - ref_out.astype(np.int16))
            mse = float(np.mean(diff.astype(np.float64) ** 2))
            parity = {"parity_on_workload": dims_ok and payload_ok and int(diff.max()) == 0,
                      "blocks_checked": int(nb), "dims_and_offsets_equal": dims_ok, "payload_bytes_equal": payload_ok,
                      "decoded_max_abs_diff_lsb": int(diff.max()), "decoded_psnr_db": None if mse == 0 else round(10 * np.log10(255.0 ** 2 / mse), 2),
                      "stored_values_max_abs_diff": float(np.max(np.abs(descs["value"][:nb].astype(np.float64) - ref_s.descs["value"]))),
                      "what": f"frame 0 of the timed workload, top {CPU_SAMPLE_ROWS} rows: GPU descriptors / payload / decoded pixels against the CPU oracle run of cpu_baseline"}

        # ---- informative: the opt-in fused-multiply-add resample (pixels within +-1 LSB of the reference, the tolerance
        # BASELINE.json states; tests/test_gpu_parity.py checks it).  Single stream; not the headline.
        fused_info = None
        if rank == 0:
            ctx.set_fast_resample(True)
            for _ in range(2):
                pl = wrapped[0][0].shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
                pl.expand_to_image(FILTER_UP, wrapped_out[0])
                pl.free()
            ctx.profile_enable(True)
            for i in range(2 * distinct):
                pl = wrapped[0][i % distinct].shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
                pl.expand_to_image(FILTER_UP, wrapped_out[0])
                pl.free()
            stream.synchronize()
            fprof = ctx.profile_read()
            ctx.profile_enable(False)
            ctx.set_fast_resample(False)
            fused_info = {"note": "pxz_ctx_set_fast_resample(1): taps as one fused multiply-add, pixels within +-1 LSB; single stream",
                          "kernel_us": {k: round(ms / n * 1e3, 2) for k, (ms, n) in fprof.items() if n}}
            fused_info["MPps_single_stream"] = round(IMG_W * IMG_H / 1e6 / (sum(fused_info["kernel_us"].values()) * 1e-6), 1)

        # ---- informative: the directional (Sobel) metric on the same frames (shrink_directionally, pixlzr.rs:187-205) ----
        sobel_info = None
        if rank == 0:
            for _ in range(2):
                pl = wrapped[0][0].shrink(BS, BS, N.METRIC_SOBEL_DIR, 8.0, FILTER_DOWN, 0)
                pl.free()
            ctx.profile_enable(True)
            for i in range(2 * distinct):
                pl = wrapped[0][i % distinct].shrink(BS, BS, N.METRIC_SOBEL_DIR, 8.0, FILTER_DOWN, 0)
                pl.expand_to_image(FILTER_UP, wrapped_out[0])
                pl.free()
            stream.synchronize()
            sprof = ctx.profile_read()
            ctx.profile_enable(False)
            sobel_info = {"note": "metric = directional Sobel, factor 8, Lanczos3 both ways; single stream",
                          "kernel_us": {k: round(ms / n * 1e3, 2) for k, (ms, n) in sprof.items() if n}}
            if "analyze_sobel" in sobel_info["kernel_us"]:
                us = sobel_info["kernel_us"]["analyze_sobel"]
                sobel_info["analyze_sobel_frac_of_hbm_peak"] = round((4 * IMG_W * IMG_H + 8 * nblocks) / (us * 1e-6) / 1e9 /
                                                                     float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
                                                                     if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 0.0, 4)

        # ---- e2e: same work through the C ABI with pinned host buffers ---------------------------------
        # `--e2e-workers` host threads, each with its own context (= its own stream) and pinned staging buffers, take
        # the frames of the step in turn, so one frame's H2D overlaps another's kernels and D2H (PCIe is full duplex).
        img_bytes = IMG_W * IMG_H * 4
        n_workers = max(1, min(args.e2e_workers, batch))
        np_imgs = [t.numpy() for t in host_imgs]

        class Worker:
            def __init__(self):
                self.ctx = N.Context(local_rank)
                self.pin = [torch.empty(nblocks * 16, dtype=torch.uint8).pin_memory(),
                            torch.empty(img_bytes, dtype=torch.uint8).pin_memory(),
                            torch.empty((IMG_H, IMG_W, 4), dtype=torch.uint8).pin_memory()]
                self.descs = self.pin[0].numpy().view(N.DESC_DTYPE)
                self.pixels, self.out = self.pin[1].numpy(), self.pin[2].numpy()
                self.h2d = self.d2h = 0

            def encode_decode(self, a):
                c = self.ctx
                im = c.image_upload(a)                                                  # H2D image
                pl = im.shrink(BS, BS, N.METRIC_OKLAB_MAD, FACTOR, FILTER_DOWN, 0)
                nbytes = pl.download_into(self.descs, self.pixels)                      # D2H descs + payload (encode result)
                pl.free()
                im.free()
                pl2 = c.payload_upload(IMG_W, IMG_H, BS, BS, 4, self.descs, self.pixels[:nbytes])  # H2D payload
                pl2.expand_into(FILTER_UP, self.out)                                    # D2H decoded image
                pl2.free()
                self.h2d += img_bytes + nbytes + nblocks * 16
                self.d2h += nbytes + nblocks * 16 + img_bytes

        workers = [Worker() for _ in range(n_workers)]

        def run_steps(k: int):
            # worker w takes frames w, w + n_workers, ... of every step; steps run back to back (no per-step join)
            def loop(wi: int):
                for _ in range(k):
                    for i in range(wi, batch, n_workers):
                        workers[wi].encode_decode(np_imgs[i % distinct])
            th = [threading.Thread(target=loop, args=(wi,)) for wi in range(n_workers)]
            for t in th:
                t.start()
            for t in th:
                t.join()

        e2e_steps = max(1, min(args.steps, args.e2e_steps))
        run_steps(1)
        for wk in workers:
            wk.h2d = wk.d2h = 0
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        run_steps(e2e_steps)
        e2e_s = time.perf_counter() - t0
        h2d = sum(wk.h2d for wk in workers)
        d2h = sum(wk.d2h for wk in workers)
        # the ceiling of that path: the same bytes of one step as plain pinned copies, both directions at once
        pcie = None
        if args.pcie_probe:
            src_pin, dst_pin = workers[0].pin[2], workers[0].pin[1]
            dbuf = torch.empty(img_bytes, dtype=torch.uint8, device=dev)
            dbuf2 = torch.empty(img_bytes, dtype=torch.uint8, device=dev)
            s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            tp0 = time.perf_counter()
            for _ in range(4):
                with torch.cuda.stream(s_up):
                    dbuf.copy_(src_pin.view(-1)[:img_bytes], non_blocking=True)
                with torch.cuda.stream(s_dn):
                    dst_pin.copy_(dbuf2, non_blocking=True)
            torch.cuda.synchronize()
            tp = time.perf_counter() - tp0
            pcie = {"h2d_plus_d2h_GBps": round(8 * img_bytes / tp / 1e9, 1), "what": "4 x (132.7 MB up + 132.7 MB down) pinned, two streams, all ranks at once"}
        for wk in workers:
            del wk.pin
        del workers

    # ---- the sharded configurations, on the same ranks ---------------------------------------------------------------
    sharded = batch_c5 = nccl_parity = None
    if not args.skip_extras:
        torch.cuda.synchronize()
        del dev_imgs, outs, wrapped, wrapped_out
        torch.cuda.empty_cache()
        with torch.cuda.stream(stream):
            try:
                sharded = run_sharded_c4(torch, dist, N, S, args, rank, world, local_rank, dev)
            except Exception as e:  # a missing block is reported, it does not take the headline down
                sharded = {"error": repr(e)}
            try:
                batch_c5 = run_batch_c5(torch, dist, N, S, args, rank, world, local_rank, dev)
            except Exception as e:
                batch_c5 = {"error": repr(e)}
            if world > 1:
                try:
                    nccl_parity = run_nccl_parity(torch, dist, N, S, None, rank, world, local_rank, dev)
                except Exception as e:
                    nccl_parity = {"error": repr(e)}

    # ---- reduce over ranks: max time -------------------------------------------------------------------
    names = ClockSampler.NAMES
    reason_bits = sum(1 << i for i, n in enumerate(names) if n in (clocks.get("reasons") or []))
    times = torch.tensor([elapsed_ms, e2e_s * 1e3, (t_launched - t_wall0) * 1e3, clocks.get("sm_mhz") or -1.0, float(reason_bits),
                          solo_plain_ms, float(host_numa.get("node", -1)), 1.0 if host_numa.get("bound") else 0.0],
                         dtype=torch.float64, device=dev)
    per_rank_ms = [elapsed_ms / args.steps]
    per_rank_e2e = [batch * e2e_steps * IMG_W * IMG_H / 1e6 / e2e_s]
    per_rank_issue = [(t_launched - t_wall0) * 1e3 / args.steps]
    per_rank_solo = [solo_plain_ms / solo_steps]
    if world > 1:
        gathered = [torch.zeros_like(times) for _ in range(world)]
        dist.all_gather(gathered, times)
        per_rank_ms = [float(t[0]) / args.steps for t in gathered]  # which rank sets the max
        per_rank_e2e = [batch * e2e_steps * IMG_W * IMG_H / 1e6 / (float(t[1]) / 1e3) for t in gathered]
        per_rank_issue = [float(t[2]) / args.steps for t in gathered]
        per_rank_solo = [float(t[5]) / solo_steps for t in gathered]
        host_numa["node_per_rank"] = [int(t[6]) for t in gathered]
        host_numa["bound_per_rank"] = [bool(t[7]) for t in gathered]
        mhz = [float(t[3]) for t in gathered]
        bits = 0
        for t in gathered:
            bits |= int(t[4])
        clocks["sm_mhz_per_rank"] = mhz
        if all(m > 0 for m in mhz):
            clocks["sm_mhz"] = min(mhz)
        clocks["reasons"] = sorted(set(clocks.get("reasons") or []) | {n for i, n in enumerate(names) if bits >> i & 1})
        head = times[:3].clone()
        dist.all_reduce(head, op=dist.ReduceOp.MAX)
        times[:3] = head
    elapsed_ms, e2e_ms, host_issue_ms = float(times[0]), float(times[1]), float(times[2])
    if world > 1:  # whole-job launch count
        lt = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(lt)
        launches = int(lt.item())
    mp_per_step = world * batch * IMG_W * IMG_H / 1e6
    value = mp_per_step * args.steps / (elapsed_ms / 1e3)
    e2e_value = mp_per_step * e2e_steps / (e2e_ms / 1e3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "6650 GB/s (of fallback)"
        n_px = IMG_W * IMG_H
        mean_payload = float(np.mean(payload_bytes))
        # algorithmic bytes per launch of every kernel (DESIGN.md "algorithmic bytes"); the guard-band recompute only
        # touches the banded tiles (about 1 %), so it gets no bandwidth figure
        algo = {
            "analyze_mad_fast": 4 * n_px + 5 * nblocks,
            "mad_exact": None,
            "plan": 4 * nblocks + 20 * nblocks,
            "resample_down": 4 * n_px + mean_payload + 20 * nblocks,
            "resample_up": mean_payload + 20 * nblocks + 4 * n_px,
        }
        kernels = {}
        for name, (ms, n) in prof.items():
            if n:
                us = ms / n * 1e3
                a = algo.get(name)
                kernels[name] = {"us": round(us, 2), "launches": int(n), "share": round(ms / solo_ms, 4)}
                if a:
                    gbs = a / (us * 1e-6) / 1e9
                    kernels[name].update({"algo_GBps": round(gbs, 1), "frac": round(gbs / peak, 4)})
        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        except OSError:
            pass
        with_bw = [k for k in kernels if "frac" in kernels[k]]
        dom = max(with_bw, key=lambda k: kernels[k]["us"] * kernels[k]["launches"]) if with_bw else None
        roofline = None
        if dom:
            roofline = {"kernel": dom, "bound": "hbm", "achieved": kernels[dom]["algo_GBps"], "peak": peak,
                        "unit": "GB/s", "frac": kernels[dom]["frac"], "traffic": traffic.get(dom),
                        "traffic_source": "profiles/r02_traffic.json (ncu --set full capture of the same workload)" if dom in traffic else None,
                        "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": int(algo[dom]), "avg_launch_us": kernels[dom]["us"],
                        "timing": "CUDA events around every launch; single-stream pass over the same frames right after the timed region "
                                  "(in the multi-stream timed region kernels of different frames overlap)",
                        "single_stream_value_MPps": round(batch * IMG_W * IMG_H / 1e6 * solo_steps / (solo_plain_ms / 1e3), 1)}
        # whole stages against the roofline, the frame counted ONCE per stage (SURVEY 8d): encode = frame read + payload and
        # descriptors written; decode = payload and descriptors read + frame written
        enc_bytes = 4 * n_px + mean_payload + 16 * nblocks
        dec_bytes = mean_payload + 16 * nblocks + 4 * n_px
        enc_us = sum(kernels[k]["us"] for k in ("analyze_mad_fast", "mad_exact", "plan", "resample_down") if k in kernels)
        dec_us = kernels.get("resample_up", {}).get("us", 0.0)
        per_image_s = elapsed_ms / 1e3 / (args.steps * batch)
        stage = {"algorithmic_bytes_per_image": int(enc_bytes + dec_bytes),
                 "GBps": round((enc_bytes + dec_bytes) / per_image_s / 1e9, 1),
                 "frac_of_hbm_peak": round((enc_bytes + dec_bytes) / per_image_s / 1e9 / peak, 4),
                 "payload_fraction": round(mean_payload / (4 * n_px), 4),
                 "encode_stage_frac": round(enc_bytes / (enc_us * 1e-6) / 1e9 / peak, 4) if enc_us else None,
                 "decode_stage_frac": round(dec_bytes / (dec_us * 1e-6) / 1e9 / peak, 4) if dec_us else None,
                 "encode_stage_us_single_stream": round(enc_us, 2), "decode_stage_us_single_stream": round(dec_us, 2),
                 "note": "frac_of_hbm_peak: the timed multi-stream region; encode / decode_stage_frac: sums of the per-launch times of the "
                         "single-stream pass, the frame counted once per stage"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args), "streams_per_gpu": n_streams,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d // e2e_steps),
                    "d2h_bytes_per_step": int(d2h // e2e_steps), "steps": e2e_steps,
                    "host_threads": n_workers, "host_numa": host_numa, "per_rank_MPps": [round(x, 1) for x in per_rank_e2e], "pcie_ceiling": pcie,
                    "path": "pxz_image_upload -> pxz_shrink -> pxz_payload_download -> pxz_payload_upload -> pxz_expand, pinned host buffers"},
            "gpu_launches": int(launches),
            "issue": {"mode": issue_mode, "note": graph_note,
                      "what": "graph = the K timed steps are captured once (same C-ABI calls, same streams) and the timed region is one "
                              "replay of that CUDA graph; direct = the Python loop issues them inside the timed region"},
            # host wall time to issue one step's launches (per rank): the step is launch-bound when this nears ms_per_step
            "host_issue_ms_per_step": round(host_issue_ms / args.steps, 4),
            "host_issue_ms_per_step_per_rank": [round(x, 4) for x in per_rank_issue],
            "ms_per_step_per_rank": [round(x, 4) for x in per_rank_ms],
            # the same frames on ONE stream per rank (no overlap between frames): tells a slow GPU from stream contention
            "single_stream_ms_per_step_per_rank": [round(x, 4) for x in per_rank_solo],
            "parity": parity,
            "fused_resample_mode": fused_info,
            "sobel_metric": sobel_info,
            "roofline": roofline,
            "kernels": kernels,
            "encode_decode_stage": stage,
            "sharded": sharded,
            "batch": batch_c5,
            "nccl_parity": nccl_parity,
            "bench_wall_s": round(time.time() - t_start, 1),
        }
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="8K frames per rank per step")
    ap.add_argument("--distinct", type=int, default=4, help="different 8K frames per rank (taken in turn)")
    ap.add_argument("--streams", type=int, default=4, help="contexts / CUDA streams of the device-resident leg")
    ap.add_argument("--issue", default="graph", choices=["graph", "direct"],
                    help="timed region: replay of a CUDA graph captured from the K steps (default) or the plain issue loop")
    ap.add_argument("--e2e-workers", type=int, default=4, help="host threads (contexts) of the end-to-end leg")
    ap.add_argument("--e2e-steps", type=int, default=2, help="steps of the end-to-end leg")
    ap.add_argument("--no-pcie-probe", dest="pcie_probe", action="store_false")
    ap.add_argument("--no-numa-bind", dest="numa_bind", action="store_false",
                    help="leave the host threads and pinned buffers wherever the OS puts them")
    ap.add_argument("--skip-extras", action="store_true", help="only the C3 headline: no sharded (C4) / batch (C5) blocks")
    ap.add_argument("--c4-side", type=int, default=65536)
    ap.add_argument("--c5-images", type=int, default=4096)
    ap.add_argument("--c5-stack", type=int, default=64, help="frames per pxz_shrink_batch call")
    ap.add_argument("--extra-reps", type=int, default=2, help="timed repetitions of the C4 / C5 passes")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 implementation")
    args.warmup = max(args.warmup, 0)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world == 1 and args.gpus > 1:
        # convenience: relaunch under torchrun when started plainly with --gpus N
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29511"), __file__] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
