"""Wrapped images (pxz_image_wrap / pxz_image_wrap_batch) of every layout the wrap accepts, through every entry point.

The kernels are chosen from the layout: base and pitch multiples of 16 (tensor copies, warp-per-tile and fast CTA-per-tile
kernels), multiples of 4 (CTA kernels that move 32-bit pixels), anything else (byte-addressed analysis; shrinking or expanding
such an RGBA view is refused), and W % 4.  Each view lives in one flat CUDA buffer: a front guard, the rows with their padding,
a back guard, every byte outside the view's pixels filled with seeded sentinel bytes.  After each call the view's pixels are
compared with the CPU oracle on the same pixels, and every byte outside them with its sentinel: a store past a trailing tile's
right edge, or a padding byte that reaches a value or a pixel, fails here even though it stays inside the allocation."""
import functools
import os

import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P
from test_gpu_parity import assert_same_payload, fast_tol, rel_close, synth
from test_quality_host import block_error

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
N = P.native

GUARD = 256
MAD, SOBEL = N.METRIC_OKLAB_MAD, N.METRIC_SOBEL_DIR
FACTOR = {MAD: 1.0, SOBEL: 6.0}
# RGBA layouts: name -> (base address mod 16, pitch of a w-pixel row)
RGBA_LAYOUTS = {
    "tight": (0, lambda w: w * 4),
    "padded16": (0, lambda w: w * 4 + 48),
    "padded4": (0, lambda w: w * 4 + 4),
    "offset4": (4, lambda w: w * 4 + 16),
    "offset8": (8, lambda w: w * 4 + 16),
    "offset12": (12, lambda w: w * 4 + 16),
}
ODD = (1, lambda w: w * 4 + 3)
# (w, h, block size): trailing tiles on both axes; 260 wide runs the RGBA fast kernels on 16-byte layouts, 259 never does
GEOMS = [(260, 132, 64), (260, 132, 32), (259, 130, 64), (259, 130, 32)]


# ---- images and oracle results, cached per image ---------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def image(w, h, c, seed=2):
    """opaque except for a translucent corner (both alpha paths), even seed"""
    img = synth(w, h, c, seed)
    if c == 4:
        img[: h // 2, : w // 3, 3] = img[: h // 2, : w // 3, 0] // 2 + 60
    img.setflags(write=False)
    return img


@functools.lru_cache(maxsize=None)
def ref_analyze(w, h, c, bs, metric, seed=2):
    return O.analyze(image(w, h, c, seed), bs, bs, metric, nthreads=8)


@functools.lru_cache(maxsize=None)
def ref_shrink(w, h, c, bs, metric, fd, fir=False, strategy=False, seed=2):
    img = image(w, h, c, seed)
    with O.resize_semantics(O.FIR if fir else O.IMAGE_RS):
        if strategy:
            return O.shrink_strategy(img, bs, bs, metric, FACTOR[metric], O.strategy_by_level()[0], nthreads=8)
        return O.shrink(img, bs, bs, metric, FACTOR[metric], fd, nthreads=8)


@functools.lru_cache(maxsize=None)
def ref_expand(w, h, c, bs, metric, fd, fu, fir=False, strategy=False, seed=2):
    ref = ref_shrink(w, h, c, bs, metric, fd, fir, strategy, seed)
    with O.resize_semantics(O.FIR if fir else O.IMAGE_RS):
        if strategy:
            return O.expand_strategy(ref, O.strategy_by_level()[1], nthreads=8)
        return O.expand(ref, fu, nthreads=8)


def upload_ref(ctx, ref):
    return ctx.payload_upload(ref.width, ref.height, ref.block_width, ref.block_height, ref.channels, ref.descs.astype(N.DESC_DTYPE),
                              ref.payload)


# ---- guarded views -----------------------------------------------------------------------------------------------------
class Guarded:
    """A view of `pixels` ([h, w, c], or [n, h, w, c] for a batch) at base address = base_mod (mod 16) with row pitch `pitch`,
    inside one flat uint8 CUDA buffer with at least GUARD sentinel bytes before and after it."""

    def __init__(self, ctx, pixels, pitch, base_mod, seed):
        self.ctx, self.batch = ctx, pixels.ndim == 4
        self.n = pixels.shape[0] if self.batch else 1
        self.h, self.w, self.c = pixels.shape[-3:]
        self.pitch = pitch
        rows = self.n * self.h
        self.buf = torch.empty(GUARD + 16 + (rows - 1) * pitch + self.w * self.c + GUARD, dtype=torch.uint8, device="cuda")
        self.off = GUARD + (base_mod - (self.buf.data_ptr() + GUARD)) % 16
        self.idx = self.off + np.arange(rows)[:, None] * pitch + np.arange(self.w * self.c)[None, :]
        self.outside = np.ones(self.buf.numel(), bool)
        self.outside[self.idx.reshape(-1)] = False
        self.fill(pixels, seed)
        ptr = self.buf.data_ptr() + self.off
        self.img = (ctx.image_wrap_batch(ptr, self.w, self.h, self.c, pitch, self.n) if self.batch
                    else ctx.image_wrap(ptr, self.w, self.h, self.c, pitch))

    def fill(self, pixels, seed):
        """sentinels from `seed` everywhere, then the view's rows"""
        self.host = np.random.default_rng(seed).integers(0, 256, self.buf.numel(), dtype=np.uint8)
        self.host[self.idx] = np.asarray(pixels).reshape(self.idx.shape)
        self.buf.copy_(torch.from_numpy(self.host))
        torch.cuda.synchronize()  # the copy runs on torch's stream, the library on the context's

    def refill(self, seed):
        """new sentinels around the same pixels"""
        self.fill(self.host[self.idx], seed)

    def read(self):
        self.ctx.synchronize()
        return self.buf.cpu().numpy()

    def assert_guards(self, data):
        bad = np.flatnonzero((data != self.host) & self.outside)
        if bad.size:
            o = int(bad[0]) - self.off
            where = "front guard" if o < 0 else (f"padding of row {o // self.pitch}" if o // self.pitch < self.n * self.h else "back guard")
            raise AssertionError(f"{bad.size} bytes outside the view changed, the first in the {where} (view offset {o})")

    def pixels(self, data):
        return data[self.idx].reshape((self.n, self.h, self.w, self.c) if self.batch else (self.h, self.w, self.c))

    def check(self, want, tol=0, what=""):
        """the view holds `want` (within tol), nothing outside it changed"""
        data = self.read()
        self.assert_guards(data)
        got = self.pixels(data)
        if tol == 0:
            assert np.array_equal(got, want), what
        else:
            assert np.abs(got.astype(np.int16) - want).max() <= tol, what

    def assert_untouched(self, what=""):
        assert np.array_equal(self.read(), self.host), f"a read-only call wrote into the source buffer {what}"

    def free(self):
        self.ctx.synchronize()
        self.img.free()


def guarded_source(ctx, img, layout, seed=101):
    base, pitch = layout
    return Guarded(ctx, img, pitch(img.shape[-2]), base, seed)


def guarded_output(ctx, w, h, c, layout, n=None, seed=202):
    """an output view whose pixels start as noise, so that a pixel the call does not write is caught too"""
    base, pitch = layout
    shape = (h, w, c) if n is None else (n, h, w, c)
    return Guarded(ctx, np.random.default_rng(seed + 1).integers(0, 256, shape, dtype=np.uint8), pitch(w), base, seed)


def _ctx_env(kind):
    old = os.environ.get("PXZ_RESAMPLE_KERNELS")
    os.environ["PXZ_RESAMPLE_KERNELS"] = kind
    try:
        return N.Context(0)
    finally:
        if old is None:
            del os.environ["PXZ_RESAMPLE_KERNELS"]
        else:
            os.environ["PXZ_RESAMPLE_KERNELS"] = old


@pytest.fixture(scope="module")
def ctxs():
    c = {"auto": N.Context(0), "warp": _ctx_env("warp"), "cta": _ctx_env("cta"), "fast": N.Context(0), "fir": N.Context(0),
         "strategy": N.Context(0)}
    c["fast"].set_fast_resample(True)
    c["fir"].set_resize_semantics(N.RESIZE_FIR)
    c["strategy"].set_strategy(*N.strategy_by_level())
    return c


# ---- analysis ----------------------------------------------------------------------------------------------------------
def analyses(view, bs):
    fast, _ = view.img.analyze(bs, bs, MAD, 0)
    exact, _ = view.img.analyze(bs, bs, MAD, N.FLAG_EXACT_VALUES)
    hz, vr = view.img.analyze(bs, bs, SOBEL, 0)
    return fast, exact, hz, vr


def assert_analyses(view, w, h, c, bs):
    fast, exact, hz, vr = got = analyses(view, bs)
    want, _ = ref_analyze(w, h, c, bs, MAD)
    whz, wvr = ref_analyze(w, h, c, bs, SOBEL)
    assert np.array_equal(exact.view("<u4"), want.view("<u4")), "Oklab-MAD exact"
    assert rel_close(fast, want, abs_=fast_tol(bs * bs)), "Oklab-MAD fast"
    assert np.array_equal(hz.view("<u4"), whz.view("<u4")) and np.array_equal(vr.view("<u4"), wvr.view("<u4")), "Sobel"
    view.assert_untouched("(analysis)")
    # other bytes around the same pixels give the same values, bit for bit: no padding byte reaches a value
    view.refill(seed=999)
    again = analyses(view, bs)
    for a, b in zip(got, again):
        assert np.array_equal(a.view("<u4"), b.view("<u4")), "a padding or guard byte changed a value"
    view.assert_untouched("(analysis, second sentinels)")


@pytest.mark.parametrize("layout", sorted(RGBA_LAYOUTS) + ["odd"])
@pytest.mark.parametrize("w,h,bs", GEOMS)
def test_rgba_analysis(ctxs, layout, w, h, bs):
    v = guarded_source(ctxs["auto"], image(w, h, 4), RGBA_LAYOUTS.get(layout, ODD))
    assert_analyses(v, w, h, 4, bs)
    v.free()


# ---- shrink ------------------------------------------------------------------------------------------------------------
def shrink_cases(bs):
    """(metric, flags, filter): both metrics, default and exact flags, the five filters in turn"""
    return [(m, fl, (i * 2 + j + bs) % 5) for i, m in enumerate((MAD, SOBEL)) for j, fl in enumerate((0, N.FLAG_EXACT_VALUES))]


@pytest.mark.parametrize("layout", sorted(RGBA_LAYOUTS))
@pytest.mark.parametrize("w,h,bs", GEOMS)
def test_rgba_shrink(ctxs, layout, w, h, bs):
    ctx = ctxs["auto"]
    v = guarded_source(ctx, image(w, h, 4), RGBA_LAYOUTS[layout])
    for metric, flags, fd in shrink_cases(bs):
        pl = v.img.shrink(bs, bs, metric, FACTOR[metric], fd, flags)
        descs, px = pl.download()
        pl.free()
        assert_same_payload(descs, px, ref_shrink(w, h, 4, bs, metric, fd), exact_values=bool(flags) or metric == SOBEL,
                            scale=10 * FACTOR[metric])
        v.assert_untouched(f"(shrink {metric} {flags})")
        v.refill(seed=fd + 7)
        pl = v.img.shrink(bs, bs, metric, FACTOR[metric], fd, flags)
        d2, p2 = pl.download()
        pl.free()
        assert np.array_equal(d2.view(np.uint8), descs.view(np.uint8)) and np.array_equal(p2, px), "a padding byte reached the payload"
        v.assert_untouched(f"(shrink {metric} {flags}, second sentinels)")
    v.free()


# ---- expand ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["auto", "warp", "cta", "fast", "fir", "strategy"])
@pytest.mark.parametrize("layout", sorted(RGBA_LAYOUTS))
@pytest.mark.parametrize("w,h,bs", GEOMS)
def test_rgba_shrink_and_expand_per_context(ctxs, kind, layout, w, h, bs):
    """shrink from a guarded source and expand into a guarded output of the same layout, on each kind of context"""
    ctx, lay = ctxs[kind], RGBA_LAYOUTS[layout]
    src = guarded_source(ctx, image(w, h, 4), lay)
    out = guarded_output(ctx, w, h, 4, lay)
    fir, strat = kind == "fir", kind == "strategy"
    flags = N.FLAG_EXACT_VALUES if kind in ("cta", "fir") else 0
    ref = ref_shrink(w, h, 4, bs, MAD, 4, fir, strat)
    pl = src.img.shrink(bs, bs, MAD, 1.0, 4, flags)
    descs, px = pl.download()
    src.assert_untouched()
    if kind == "fast":  # fused multiply-add: +-1 LSB; the decode of the oracle's payload then differs by +-1 too
        assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"])
        assert np.array_equal(descs["offset"], ref.descs["offset"])
        assert np.abs(px.astype(np.int16) - ref.payload).max() <= 1
        pl.free()
        pl = upload_ref(ctx, ref)
    else:
        assert_same_payload(descs, px, ref, exact_values=bool(flags), scale=10.0)
    for fu in ([4] if strat else range(5)):  # with a strategy the filters come from the table
        pl.expand_to_image(fu, out.img)
        out.check(ref_expand(w, h, 4, bs, MAD, 4, fu, fir, strat), tol=1 if kind == "fast" else 0, what=f"filter {fu}")
    pl.free()
    src.free()
    out.free()


# ---- regions and quadtree ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", sorted(RGBA_LAYOUTS))
@pytest.mark.parametrize("w,h,bs", GEOMS)
def test_rgba_region_into_guarded_view(ctxs, layout, w, h, bs):
    ctx, lay = ctxs["auto"], RGBA_LAYOUTS[layout]
    ref = ref_shrink(w, h, 4, bs, MAD, 4)
    pl = upload_ref(ctx, ref)
    # block-aligned to the image's end (expands in place) and unaligned (staged, then copied)
    for i, (x, y, rw, rh) in enumerate([(bs, bs, w - bs, h - bs), (5, 3, w - 13, h - 7)]):
        for fu in (i, 4 - i):
            out = guarded_output(ctx, rw, rh, 4, lay, seed=300 + fu)
            pl.expand_region_to_image(fu, x, y, rw, rh, out.img)
            out.check(ref_expand(w, h, 4, bs, MAD, 4, fu)[y:y + rh, x:x + rw], what=f"rect {x, y, rw, rh} filter {fu}")
            out.free()
    pl.free()


@pytest.mark.parametrize("layout", sorted(RGBA_LAYOUTS))
@pytest.mark.parametrize("w,h,bs", GEOMS)
def test_rgba_tree_process_into_guarded_view(ctxs, layout, w, h, bs):
    ctx, lay = ctxs["auto"], RGBA_LAYOUTS[layout]
    img = image(w, h, 4)
    src = guarded_source(ctx, img, lay)
    out = guarded_output(ctx, w, h, 4, lay)
    fd, fu = bs % 5, (bs + 2) % 5
    src.img.tree_process(0.02, bs, bs, 4, 4, fd, fu, out.img)
    want = O.tree_process(img, 0.02, bs, bs, 4, 4, fd, fu)
    out.check(want)
    assert not np.array_equal(want, img)  # something was reduced
    src.assert_untouched()
    src.free()
    out.free()


# ---- the rate calls read the source as the shrink does -----------------------------------------------------------------
@pytest.mark.parametrize("layout", ["padded16", "padded4"])
@pytest.mark.parametrize("w,h,bs", [(260, 132, 64), (259, 130, 32)])
def test_rate_calls_on_wrapped_sources_equal_uploads(ctxs, layout, w, h, bs):
    ctx = ctxs["auto"]
    img = image(w, h, 4)
    src = guarded_source(ctx, img, RGBA_LAYOUTS[layout])
    up = ctx.image_upload(img)

    def calls(x):
        out = [*x.rd_curve(bs, bs, MAD, 2, 4), *x.rd_curve(bs, bs, SOBEL, 4, 1), *x.rdo_curve(bs, bs, 4, 4),
               *x.strategy_measure(bs, bs, MAD, 0.2)]
        fast = None
        for flags in (0, N.FLAG_EXACT_VALUES):
            pl, k = x.shrink_to_size(bs, bs, MAD, w * h, 4, flags)
            descs, px = pl.download()
            pl.free()
            out += [np.float32(k), descs["w"], descs["h"], descs["offset"], px]
            # without EXACT_VALUES the stored values are the fast kernel's, and padded4 runs another one than the upload
            if flags:
                out.append(descs["value"])
            else:
                fast = descs["value"], k
        return out, fast

    (a_all, (a_fast, k)), (b_all, (b_fast, _)) = calls(src.img), calls(up)
    for a, b in zip(a_all, b_all):
        # bit patterns: descriptor fields are strided views of the descriptor records
        a, b = np.ascontiguousarray(np.atleast_1d(a)), np.ascontiguousarray(np.atleast_1d(b))
        assert a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))
    assert rel_close(a_fast, b_fast, abs_=2 * fast_tol(bs * bs, 15.0 * k))  # each within fast_tol of the reference order
    src.assert_untouched()
    up.free()
    src.free()


# ---- batches -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["auto", "warp", "cta"])
@pytest.mark.parametrize("layout", ["padded16", "padded4"])
@pytest.mark.parametrize("w,h,bs", [(260, 132, 64), (259, 130, 32)])
def test_batch_of_wrapped_images(ctxs, kind, layout, w, h, bs):
    ctx, lay = ctxs[kind], RGBA_LAYOUTS[layout]
    seeds = (2, 4, 6)
    src = guarded_source(ctx, np.stack([image(w, h, 4, s) for s in seeds]), lay)
    out = guarded_output(ctx, w, h, 4, lay, n=3)
    pl = src.img.shrink(bs, bs, MAD, 1.0, 4, 0)
    descs, px = pl.download()
    src.assert_untouched()
    per, off = len(descs) // 3, 0
    for i, s in enumerate(seeds):
        ref = ref_shrink(w, h, 4, bs, MAD, 4, seed=s)
        d = descs[i * per:(i + 1) * per].copy()
        d["offset"] -= off
        assert_same_payload(d, px[off:off + ref.payload.size], ref, exact_values=False, scale=10.0)
        off += ref.payload.size
    for fu in (0, 4):
        pl.expand_to_image(fu, out.img)
        out.check(np.stack([ref_expand(w, h, 4, bs, MAD, 4, fu, seed=s) for s in seeds]), what=f"filter {fu}")
    pl.free()
    src.free()
    out.free()


# ---- RGB: any layout, both the RGBA kernels (W % 4 == 0, via widen / narrow) and the 3-channel kernels -------------------
@pytest.mark.parametrize("extra", [0, 1, 5])
@pytest.mark.parametrize("base", [0, 1, 2, 3])
@pytest.mark.parametrize("w,h,bs", [(260, 132, 64), (259, 130, 32)])
def test_rgb_layouts(ctxs, base, extra, w, h, bs):
    ctx = ctxs["auto"]
    lay = (base, lambda x: x * 3 + extra)
    img = image(w, h, 3)
    src = guarded_source(ctx, img, lay)
    assert_analyses(src, w, h, 3, bs)
    for metric, flags, fd in shrink_cases(bs):
        pl = src.img.shrink(bs, bs, metric, FACTOR[metric], fd, flags)
        descs, px = pl.download()
        pl.free()
        assert_same_payload(descs, px, ref_shrink(w, h, 3, bs, metric, fd), exact_values=bool(flags) or metric == SOBEL,
                            scale=10 * FACTOR[metric])
    src.assert_untouched()
    pl = src.img.shrink(bs, bs, MAD, 1.0, 4, 0)
    out = guarded_output(ctx, w, h, 3, lay)
    for fu in range(5):
        pl.expand_to_image(fu, out.img)
        out.check(ref_expand(w, h, 3, bs, MAD, 4, fu), what=f"filter {fu}")
    for i, (x, y, rw, rh) in enumerate([(bs, bs, w - bs, h - bs), (5, 3, w - 13, h - 7)]):
        reg = guarded_output(ctx, rw, rh, 3, lay, seed=400 + i)
        pl.expand_region_to_image(2 * i, x, y, rw, rh, reg.img)
        reg.check(ref_expand(w, h, 3, bs, MAD, 4, 2 * i)[y:y + rh, x:x + rw], what=f"rect {x, y, rw, rh}")
        reg.free()
    pl.free()
    src.img.tree_process(0.02, bs, bs, 4, 4, 4, 0, out.img)
    out.check(O.tree_process(img, 0.02, bs, bs, 4, 4, 4, 0), what="tree")
    # the fir semantics run their own (byte-addressed) kernel
    fir = ctxs["fir"]
    fsrc = guarded_source(fir, img, lay)
    pl = fsrc.img.shrink(bs, bs, MAD, 1.0, 4, N.FLAG_EXACT_VALUES)
    descs, px = pl.download()
    assert_same_payload(descs, px, ref_shrink(w, h, 3, bs, MAD, 4, fir=True), exact_values=True)
    fout = guarded_output(fir, w, h, 3, lay)
    pl.expand_to_image(3, fout.img)
    fout.check(ref_expand(w, h, 3, bs, MAD, 4, 3, fir=True))
    pl.free()
    for v in (src, out, fsrc, fout):
        v.free()


# ---- RGBA views that are not 4-byte aligned: analysis and image error only -----------------------------------------------
@pytest.mark.parametrize("w,h,bs", [(260, 132, 64), (259, 130, 32)])
def test_odd_rgba_image_error(ctxs, w, h, bs):
    ctx = ctxs["auto"]
    a = image(w, h, 4)
    b = np.clip(a.astype(np.int16) + np.random.default_rng(w).integers(-9, 10, a.shape), 0, 255).astype(np.uint8)
    v = guarded_source(ctx, a, ODD)
    ub = ctx.image_upload(b)
    sse, mx, total = v.img.error(ub, bs, bs)
    want_sse, want_max = block_error(a, b, bs, bs)
    assert np.array_equal(sse, want_sse) and np.array_equal(mx, want_max) and total == int(want_sse.sum())
    v.assert_untouched()
    ub.free()
    v.free()


@pytest.mark.parametrize("w,h,bs", [(260, 132, 64), (259, 130, 32)])
def test_odd_rgba_views_refuse_every_resample(ctxs, w, h, bs):
    """Shrinking an RGBA view whose base or pitch is not a multiple of 4, or expanding into one, is refused with
    PXZ_E_UNSUPPORTED, and neither the source nor the output buffer is written."""
    ctx = ctxs["auto"]
    img = image(w, h, 4)
    src = guarded_source(ctx, img, ODD)
    out = guarded_output(ctx, w, h, 4, ODD)
    bsrc = guarded_source(ctx, np.stack([img, img]), ODD)
    bout = guarded_output(ctx, w, h, 4, ODD, n=2)
    rw, rh = w - bs, h - bs
    reg = [guarded_output(ctx, rw, rh, 4, ODD, seed=500), guarded_output(ctx, w - 13, h - 7, 4, ODD, seed=501)]
    up = ctx.image_upload(img)
    good_out = guarded_output(ctx, w, h, 4, RGBA_LAYOUTS["padded16"])
    ref = ref_shrink(w, h, 4, bs, MAD, 4)
    pl = upload_ref(ctx, ref)
    second = ref.descs.copy()
    second["offset"] += ref.payload.size  # a batch payload's offsets run through all its images
    bpl = ctx.payload_upload_batch(w, h, bs, bs, 4, 2, np.concatenate([ref.descs, second]).astype(N.DESC_DTYPE),
                                   np.concatenate([ref.payload, ref.payload]))
    s = src.img
    calls = {
        "shrink": lambda: s.shrink(bs, bs, MAD, 1.0, 4, 0),
        "shrink exact": lambda: s.shrink(bs, bs, MAD, 1.0, 4, N.FLAG_EXACT_VALUES),
        "shrink sobel": lambda: s.shrink(bs, bs, SOBEL, 6.0, 1, 0),
        "shrink fir": lambda: ctxs["fir"].image_wrap(src.buf.data_ptr() + src.off, w, h, 4, src.pitch).shrink(bs, bs, MAD, 1.0, 4, 0),
        "shrink batch": lambda: bsrc.img.shrink(bs, bs, MAD, 1.0, 4, 0),
        "shrink_to_size": lambda: s.shrink_to_size(bs, bs, MAD, w * h * 4, 4),
        "shrink_to_error": lambda: s.shrink_to_error(bs, bs, MAD, 1 << 60, 4, 4),
        "rd_curve": lambda: s.rd_curve(bs, bs, MAD, 4, 4),
        "rdo_curve": lambda: s.rdo_curve(bs, bs, 4, 4),
        "rdo_shrink_to_size": lambda: s.rdo_shrink_to_size(bs, bs, w * h * 4, 4, 4),
        "rdo_shrink_to_error": lambda: s.rdo_shrink_to_error(bs, bs, 1 << 60, 4, 4),
        "strategy_measure": lambda: s.strategy_measure(bs, bs, MAD, 0.2),
        "tree_process source": lambda: s.tree_process(0.02, bs, bs, 4, 4, 4, 0, good_out.img),
        "tree_process output": lambda: up.tree_process(0.02, bs, bs, 4, 4, 4, 0, out.img),
        "expand_to_image": lambda: pl.expand_to_image(4, out.img),
        "expand batch": lambda: bpl.expand_to_image(4, bout.img),
        "expand_region aligned": lambda: pl.expand_region_to_image(4, bs, bs, rw, rh, reg[0].img),
        "expand_region staged": lambda: pl.expand_region_to_image(4, 5, 3, w - 13, h - 7, reg[1].img),
    }
    for name, call in calls.items():
        with pytest.raises(N.PixlzrError) as e:
            call()
        assert e.value.status == N.E_UNSUPPORTED, name
    for v in (src, out, bsrc, bout, *reg, good_out):
        v.assert_untouched()
        v.free()
    pl.free()
    bpl.free()
    up.free()


# ---- a pitch so wide that a 64-row tile spans more than 4 GiB (a column strip of a very wide tensor) ---------------------
WIDE_PITCH = (1 << 26) + (1 << 22)  # 63 rows of it exceed 2^32 bytes


def test_wide_pitch_view(ctxs):
    """Oklab-MAD's fast analysis of 64x64 RGBA tiles whose last rows lie more than 2^32 bytes past the tile's first byte: the
    in-tile offsets must not wrap into the padding of the first rows (here zeros, against opaque noise)."""
    w, h, bs = 256, 64, 64
    span = (h - 1) * WIDE_PITCH + w * 4
    if torch.cuda.mem_get_info()[0] < (6 << 30):
        pytest.skip("needs 6 GB of free device memory")
    ctx = ctxs["auto"]
    rng = np.random.default_rng(17)
    img = np.concatenate([rng.integers(0, 256, (h, w, 3), dtype=np.uint8), np.full((h, w, 1), 255, np.uint8)], -1)
    buf = torch.zeros(GUARD + span + GUARD, dtype=torch.uint8, device="cuda")
    rows = buf.as_strided((h, w * 4), (WIDE_PITCH, 1), GUARD)
    rows.copy_(torch.from_numpy(img.reshape(h, w * 4)))
    torch.cuda.synchronize()
    v = ctx.image_wrap(buf.data_ptr() + GUARD, w, h, 4, WIDE_PITCH)
    want, _ = O.analyze(img, bs, bs, MAD)
    fast, _ = v.analyze(bs, bs, MAD, 0)
    exact, _ = v.analyze(bs, bs, MAD, N.FLAG_EXACT_VALUES)
    assert np.array_equal(exact.view("<u4"), want.view("<u4"))
    assert rel_close(fast, want, abs_=fast_tol(bs * bs)), (fast, want)
    ref = O.shrink(img, bs, bs, MAD, 1.0, O.LANCZOS3)
    pl = v.shrink(bs, bs, MAD, 1.0, O.LANCZOS3, 0)
    descs, px = pl.download()
    assert_same_payload(descs, px, ref, exact_values=False, scale=10.0)
    # and back into the same view
    pl.expand_to_image(O.LANCZOS3, v)
    ctx.synchronize()
    pl.free()
    v.free()
    assert np.array_equal(rows.contiguous().cpu().numpy().reshape(h, w, 4), O.expand(ref, O.LANCZOS3))
    assert not buf[:GUARD].any() and not buf[GUARD + span:].any()
    for r in range(h - 1):  # each row's padding, one contiguous slice at a time
        assert not buf[GUARD + r * WIDE_PITCH + w * 4: GUARD + (r + 1) * WIDE_PITCH].any(), r
    del rows, buf
    torch.cuda.empty_cache()


def test_handles_outliving_their_context():
    """A failed call leaves its images and payloads to the garbage collector, which may finalise their context first (a cycle
    through a traceback holds them all).  Freeing them after the context is closed only drops the handles: the library's
    free of a payload or an owned image uses its context."""
    ctx = N.Context(0)
    owned = ctx.image_upload(image(64, 48, 4))
    buf = torch.zeros(48 * 256, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    wrapped = ctx.image_wrap(buf.data_ptr(), 64, 48, 4, 256)
    pl = owned.shrink(32, 32, MAD, 1.0, 4, 0)
    ctx.close()
    for x in (pl, owned, wrapped):
        x.free()
        assert not x.handle
