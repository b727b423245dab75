"""Random access on the device: windows of payloads (pxz_payload_window) and pixel rectangles of the decoded image
(pxz_expand_region, Pixlzr.decode_vec_region_to_image / to_image_region).  Every rectangle is compared byte for byte with
the same rectangle of the whole decode of the same payload, which the parity suite pins against the oracle and the
reference's files."""
import os

import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P
from conftest import GOLDEN, load_png

pytestmark = pytest.mark.gpu
N = P.native


def synth(w, h, c, seed):
    """smooth base + per-32x32 noise of varying amplitude (many levels), translucent alpha for odd seeds"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.stack([128 + 96 * np.sin(xx / 97.0 + seed), 128 + 96 * np.cos(yy / 131.0), 128 + 64 * np.sin((xx + yy) / 61.0)], -1)
    amp = rng.choice([0, 1, 2, 4, 8, 16, 32, 64, 128], size=((h + 31) // 32, (w + 31) // 32)).astype(np.float32)
    amp = np.kron(amp, np.ones((32, 32), np.float32))[:h, :w]
    img = np.clip(base + (rng.random((h, w, 3), dtype=np.float32) - 0.5) * 2 * amp[..., None], 0, 255).astype(np.uint8)
    if c == 4:
        a = np.full((h, w, 1), 255, np.uint8) if seed % 2 == 0 else rng.integers(0, 256, (h, w, 1), dtype=np.uint8)
        img = np.concatenate([img, a], -1)
    return np.ascontiguousarray(img)


def rects(W, H, bw, bh, seed, n=8):
    """(x, y, w, h): 1x1 at every corner, block-aligned, straddling the trailing column / row, the whole image, seeded random"""
    out = [(0, 0, 1, 1), (W - 1, 0, 1, 1), (0, H - 1, 1, 1), (W - 1, H - 1, 1, 1), (0, 0, W, H),
           (bw, bh, min(2 * bw, W - bw), min(bh, H - bh)) if W > bw and H > bh else (0, 0, 1, 1),
           (max(0, W - bw - 5), max(0, H - 3 * bh // 2), min(W, bw + 5), min(H, 3 * bh // 2)),  # trailing column and row
           (W // 3, max(0, H - 7), W // 3, min(7, H)), (max(0, W - 9), H // 4, min(9, W), H // 2)]
    rng = np.random.default_rng(seed)
    for _ in range(n):
        x, y = int(rng.integers(0, W)), int(rng.integers(0, H))
        out.append((x, y, int(rng.integers(1, W - x + 1)), int(rng.integers(1, H - y + 1))))
    return out


def assert_regions(pl, filt, full, rs):
    for (x, y, w, h) in rs:
        got = pl.expand_region(filt, x, y, w, h)
        assert np.array_equal(got, full[y:y + h, x:x + w]), (filt, x, y, w, h)


def _ctx_env(**env):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return N.Context(0)
    finally:
        for k, v in old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def ctx():
    return N.Context(0)


# ---- shapes x filters, payloads from pxz_shrink --------------------------------------------------------------------
@pytest.mark.parametrize("w,h,c,bs", [
    (1920, 1080, 3, 32),   # RGB, W % 4 == 0: expands on the RGBA kernels
    (1080, 1617, 4, 64),   # trailing column (56 px) and row (17 px)
    (7680, 4320, 4, 64),   # 8K: the full decode runs the warp-per-tile kernels, small windows the CTA kernels
    (1001, 603, 3, 32),    # RGB, W % 4 != 0: the 3-channel kernels
    (500, 333, 4, 13),     # odd block size: the generic kernels
])
def test_regions_equal_the_crop_of_the_whole_decode(ctx, w, h, c, bs):
    img = synth(w, h, c, seed=w + c)
    d = ctx.image_upload(img)
    pl = d.shrink(bs, bs, N.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, 0)
    for filt in range(5):
        full = pl.expand(filt)
        assert_regions(pl, filt, full, rects(w, h, bs, bs, seed=filt, n=4 if w > 4000 else 8))
    pl.free()
    d.free()


def test_regions_sobel_and_fir_semantics(ctx):
    img = synth(452, 648, 4, seed=3)
    d = ctx.image_upload(img)
    pl = d.shrink(64, 64, N.METRIC_SOBEL_DIR, 6.0, O.CATMULLROM, 0)  # the two axes at different levels
    full = pl.expand(O.GAUSSIAN)
    assert_regions(pl, O.GAUSSIAN, full, rects(452, 648, 64, 64, seed=5))
    pl.free(); d.free()
    fir = N.Context(0)
    fir.set_resize_semantics(N.RESIZE_FIR)
    for c in (3, 4):
        img = synth(300, 230, c, seed=8 + c)
        d = fir.image_upload(img)
        pl = d.shrink(32, 32, N.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, 0)
        for filt in range(5):
            assert_regions(pl, filt, pl.expand(filt), rects(300, 230, 32, 32, seed=filt, n=3))
        pl.free(); d.free()


def test_regions_with_per_block_filters(ctx):
    """Strategy.by_level(): expand-side indices of a shrink payload (copied by the window kernel) and per-block filters of a
    payload decoded from a file (folded into its table indices)."""
    sctx = N.Context(0)
    st = P.Strategy.by_level()
    sctx.set_strategy(st.down, st.up)
    img = synth(1080, 1617, 4, seed=2)
    d = sctx.image_upload(img)
    pl = d.shrink(64, 64, N.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, 0)
    full = pl.expand(O.LANCZOS3)
    assert_regions(pl, O.LANCZOS3, full, rects(1080, 1617, 64, 64, seed=9))
    data = pl.to_container(4, True)
    pl.free(); d.free()
    pf, _ = sctx.payload_from_container(data)
    assert np.array_equal(pf.expand(O.LANCZOS3), full)
    assert_regions(pf, O.LANCZOS3, full, rects(1080, 1617, 64, 64, seed=10))
    assert np.array_equal(P.Pixlzr.decode_vec_region_to_image(data, P.FilterType.Lanczos3, 100, 1500, 900, 117, ctx=sctx),
                          full[1500:1617, 100:1000])
    pf.free()


def test_fused_mode_regions():
    """Fused arithmetic is +-1 LSB; a small window may run the other kernel family than the whole frame, so a region is
    within +-1 of the crop, and bit-exact when the family is forced the same for both."""
    img = synth(2048, 1536, 4, seed=4)
    for kind in (None, "warp", "cta"):
        c = N.Context(0) if kind is None else _ctx_env(PXZ_RESAMPLE_KERNELS=kind)
        c.set_fast_resample(True)
        d = c.image_upload(img)
        # 3072 tiles: by default the whole frame takes the warp kernels (>= 16 tiles per SM), small windows the CTA kernels
        pl = d.shrink(32, 32, N.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, 0)
        for filt in (1, 4):
            full = pl.expand(filt)
            for (x, y, w, h) in rects(2048, 1536, 32, 32, seed=filt):
                got = pl.expand_region(filt, x, y, w, h)
                ref = full[y:y + h, x:x + w]
                if kind is None:
                    assert np.abs(got.astype(np.int16) - ref).max() <= 1, (filt, x, y, w, h)
                else:
                    assert np.array_equal(got, ref), (kind, filt, x, y, w, h)
        pl.free(); d.free()


# ---- payload origins -----------------------------------------------------------------------------------------------
def test_regions_of_uploads_with_blocks_larger_than_their_tiles(ctx):
    """RGB, W % 4 == 0: the expand converts the payload to RGBA, whose buffer must hold blocks larger than their tiles."""
    rng = np.random.default_rng(5)
    w, h, bw, bh, c = 152, 100, 32, 32, 3
    cols, rows = O.grid(w, h, bw, bh)
    descs = np.zeros(cols * rows, O.DESC_DTYPE)
    parts, off = [], 0
    for i in range(cols * rows):
        sw, sh = int(rng.integers(24, 65)), int(rng.integers(24, 65))
        descs[i] = (off, 0.5, sw, sh)
        parts.append(rng.integers(0, 256, sw * sh * c, dtype=np.uint8))
        off += sw * sh * c
    payload = np.concatenate(parts)
    assert payload.size > w * h * 4  # more than even the RGBA image holds
    ref = O.Shrunk(w, h, bw, bh, c, descs, payload)
    pl = ctx.payload_upload(w, h, bw, bh, c, descs.astype(N.DESC_DTYPE), payload)
    for filt in range(5):
        full = pl.expand(filt)
        assert np.array_equal(full, O.expand(ref, filt, nthreads=8)), filt
        assert_regions(pl, filt, full, rects(w, h, bw, bh, seed=filt))
    # the host-held payload API uploads only the touched blocks
    pix = P.Pixlzr(w, h, bw, bh)
    pix._descs, pix._pixels, pix._channels, pix._values_present = descs.astype(N.DESC_DTYPE), payload, c, True
    full = pl.expand(O.CATMULLROM)
    for (x, y, rw, rh) in rects(w, h, bw, bh, seed=3):
        assert np.array_equal(pix.to_image_region(P.FilterType.CatmullRom, x, y, rw, rh), full[y:y + rh, x:x + rw])
    pl.free()


def test_regions_of_decoded_files(ctx):
    for c in (3, 4):
        img = synth(1000, 760, c, seed=20 + c)
        d = ctx.image_upload(img)
        pl = d.shrink(64, 64, N.METRIC_OKLAB_MAD, 1.0, O.TRIANGLE, 0)
        data = pl.to_container(1, True)
        pl.free(); d.free()
        pf, filt = ctx.payload_from_container(data)
        assert filt == 1
        full = pf.expand(O.LANCZOS3)
        assert_regions(pf, O.LANCZOS3, full, rects(1000, 760, 64, 64, seed=c))
        for (x, y, w, h) in rects(1000, 760, 64, 64, seed=c + 10):
            got = P.Pixlzr.decode_vec_region_to_image(memoryview(data), P.FilterType.Lanczos3, x, y, w, h, ctx=ctx)
            assert np.array_equal(got, full[y:y + h, x:x + w]), (x, y, w, h)
        pf.free()


def test_reference_artefacts():
    raw = open(os.path.join(GOLDEN, "Big-Ruscher.pix"), "rb").read()
    png = load_png("Big-Ruscher.pix.png")
    pix = P.Pixlzr.decode_from_vec(raw)
    for (x, y, w, h) in rects(1920, 1080, 32, 32, seed=1):
        want = png[y:y + h, x:x + w]
        assert np.array_equal(P.Pixlzr.decode_vec_region_to_image(raw, P.FilterType.Nearest, x, y, w, h), want), (x, y, w, h)
        assert np.array_equal(pix.to_image_region(P.FilterType.Nearest, x, y, w, h), want), (x, y, w, h)
    raw = open(os.path.join(GOLDEN, "base.pixlzr"), "rb").read()
    png = load_png("base.png")
    for (x, y, w, h) in rects(png.shape[1], png.shape[0], 64, 64, seed=2):
        got = P.Pixlzr.decode_vec_region_to_image(raw, P.FilterType.Lanczos3, x, y, w, h)
        assert np.array_equal(got, png[y:y + h, x:x + w]), (x, y, w, h)
    # from_image keeps the source: the region is its crop
    src = P.Pixlzr.from_image(png, 64, 64)
    assert np.array_equal(src.to_image_region(P.FilterType.Nearest, 5, 7, 100, 90), png[7:97, 5:105])


# ---- window payloads -----------------------------------------------------------------------------------------------
def test_window_payload_contents(ctx):
    img = synth(1080, 1617, 4, seed=6)
    d = ctx.image_upload(img)
    pl = d.shrink(64, 64, N.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, 0)
    descs, px = pl.download()
    cols, rows = N.grid(1080, 1617, 64, 64)
    data = pl.to_container(4, True)
    full = pl.expand(O.LANCZOS3)
    for (c0, r0, nc, nr) in [(0, 0, 1, 1), (cols - 1, rows - 1, 1, 1), (3, 4, 7, 9), (0, 0, cols, rows), (cols - 3, 0, 3, rows)]:
        win = pl.window(c0, r0, nc, nr)
        info = win.info()
        assert (info["w"], info["h"], info["bw"], info["bh"], info["cols"], info["rows"], info["channels"]) == \
               (min(1080, (c0 + nc) * 64) - c0 * 64, min(1617, (r0 + nr) * 64) - r0 * 64, 64, 64, nc, nr, 4)
        wd, wp = win.download()
        idx = ((r0 + np.arange(nr))[:, None] * cols + (c0 + np.arange(nc))[None, :]).reshape(-1)
        ref = descs[idx]
        sizes = ref["w"].astype(np.int64) * ref["h"] * 4
        assert np.array_equal(wd["w"], ref["w"]) and np.array_equal(wd["h"], ref["h"])
        assert np.array_equal(wd["value"].view(np.uint32), ref["value"].view(np.uint32))
        assert np.array_equal(wd["offset"], np.concatenate([[0], np.cumsum(sizes)[:-1]]))
        assert np.array_equal(wp, np.concatenate([px[o:o + n] for o, n in zip(ref["offset"].tolist(), sizes.tolist())]))
        assert win.to_container(4, True) == N.container_crop(data, c0, r0, nc, nr)
        x0, y0 = c0 * 64, r0 * 64
        assert np.array_equal(win.expand(O.LANCZOS3), full[y0:y0 + info["h"], x0:x0 + info["w"]])
        # a window of a window, and a window outliving its parent's handle
        if nc >= 2 and nr >= 2:
            ww = win.window(1, 1, nc - 1, nr - 1)
            wi = ww.info()
            assert np.array_equal(ww.expand(O.LANCZOS3), full[y0 + 64:y0 + 64 + wi["h"], x0 + 64:x0 + 64 + wi["w"]])
            ww.free()
        win.free()
    pl.free(); d.free()


@pytest.mark.parametrize("c", [3, 4])
def test_window_of_exact_shrink_is_the_shrink_of_the_crop(ctx, c):
    img = synth(1080, 1617, c, seed=12 + c)
    d = ctx.image_upload(img)
    pl = d.shrink(64, 64, N.METRIC_OKLAB_MAD, 1.0, O.CATMULLROM, N.FLAG_EXACT_VALUES)
    for (c0, r0, nc, nr) in [(2, 3, 5, 6), (16, 25, 1, 1), (10, 0, 7, 26)]:
        win = pl.window(c0, r0, nc, nr)
        crop = np.ascontiguousarray(img[r0 * 64:(r0 + nr) * 64, c0 * 64:(c0 + nc) * 64])
        dc = ctx.image_upload(crop)
        pc = dc.shrink(64, 64, N.METRIC_OKLAB_MAD, 1.0, O.CATMULLROM, N.FLAG_EXACT_VALUES)
        (wd, wp), (cd, cp) = win.download(), pc.download()
        assert np.array_equal(wd.view(np.uint8), cd.view(np.uint8)) and np.array_equal(wp, cp), (c0, r0, nc, nr)
        pc.free(); dc.free(); win.free()
    pl.free(); d.free()


# ---- errors --------------------------------------------------------------------------------------------------------
def test_region_errors(ctx):
    img = synth(300, 200, 4, seed=1)
    d = ctx.image_upload(img)
    pl = d.shrink(32, 32, N.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, 0)
    out = ctx.image_alloc(10, 10, 4)
    L = N.lib()

    def status(x, y, w, h, img_out=out, filt=4):
        return L.pxz_expand_region(ctx.handle, pl.handle, filt, x, y, w, h, img_out.handle)

    assert status(0, 0, 10, 10) == N.OK
    assert status(0, 0, 0, 10) == N.E_ARG and status(0, 0, 10, 0) == N.E_ARG          # empty
    assert status(291, 0, 10, 10) == N.E_ARG and status(0, 191, 10, 10) == N.E_ARG  # outside the image
    assert status(300, 0, 10, 10) == N.E_ARG and status(0xFFFFFFFB, 0, 10, 10) == N.E_ARG
    assert status(0, 0, 11, 10) == N.E_ARG and status(0, 0, 10, 9) == N.E_ARG       # output geometry
    rgb = ctx.image_alloc(10, 10, 3)
    assert status(0, 0, 10, 10, rgb) == N.E_ARG
    assert status(0, 0, 10, 10, filt=5) == N.E_ARG
    for bad in [(0, 0, 0, 1), (0, 0, 1, 0), (10, 0, 1, 1), (0, 7, 1, 1), (9, 0, 2, 1), (0, 6, 1, 2)]:
        with pytest.raises(N.PixlzrError) as e:
            pl.window(*bad)
        assert e.value.status == N.E_ARG, bad
    with pytest.raises(N.PixlzrError) as e:
        P.Pixlzr.decode_vec_region_to_image(pl.to_container(), P.FilterType.Nearest, 290, 0, 11, 5, ctx=ctx)
    assert e.value.status == N.E_ARG
    # batches: out of scope, refused
    batch = ctx.image_upload_batch(np.stack([img, img]))
    pb = batch.shrink(32, 32, N.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, 0)
    with pytest.raises(N.PixlzrError) as e:
        pb.window(0, 0, 1, 1)
    assert e.value.status == N.E_UNSUPPORTED
    assert L.pxz_expand_region(ctx.handle, pb.handle, 4, 0, 0, 10, 10, out.handle) == N.E_UNSUPPORTED
    pb.free(); batch.free(); out.free(); rgb.free(); pl.free(); d.free()


def test_region_into_a_wrapped_tensor(ctx):
    torch = pytest.importorskip("torch")
    img = synth(640, 480, 4, seed=2)
    d = ctx.image_upload(img)
    pl = d.shrink(64, 64, N.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, 0)
    full = pl.expand(O.LANCZOS3)
    t = torch.zeros((100, 130, 4), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()  # the fill runs on torch's stream, the region on the context's
    im = ctx.image_wrap(t.data_ptr(), 130, 100, 4, t.stride(0))
    pl.expand_region_to_image(O.LANCZOS3, 77, 301, 130, 100, im)
    ctx.synchronize()
    assert np.array_equal(t.cpu().numpy(), full[301:401, 77:207])
    im.free(); pl.free(); d.free()
