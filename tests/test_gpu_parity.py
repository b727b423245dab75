"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle and the
reference's golden files.  Bars (BASELINE.json north star): block grid, levels / dims and chosen
scales bit-exact; stored f32 values bit-exact in exact mode and within 1e-4 relative (+1e-6 abs) in
the default fast mode; resampled pixels bit-exact with the oracle (the bar is +-1 LSB)."""
import os

import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P
from conftest import GOLDEN, load_png

pytestmark = pytest.mark.gpu
N = P.native

FILTERS = [0, 1, 2, 3, 4]
# the five (down, up) pairs logged in the reference's strategies.txt
STRATEGIES = [(0, 0), (1, 0), (2, 4), (4, 2), (4, 4)]


@pytest.fixture(scope="module")
def ctx():
    return N.Context(0)


def synth(w, h, c, seed, kind="mixed"):
    """Seeded test image: smooth base + per-64x64-region noise of varying amplitude, so that block
    values spread over many levels."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.stack([128 + 96 * np.sin(xx / 9700.0 + seed), 128 + 96 * np.cos(yy / 13100.0), 128 + 64 * np.sin((xx + yy) / 6100.0)], -1)
    if kind == "flat":
        img = np.full((h, w, 3), 77.0, np.float32)
    elif kind == "noise":
        img = rng.integers(0, 256, (h, w, 3)).astype(np.float32)
    else:
        amp = rng.choice([0, 1, 2, 4, 8, 16, 32, 64, 128], size=((h + 31) // 32, (w + 31) // 32)).astype(np.float32)
        amp = np.kron(amp, np.ones((32, 32), np.float32))[:h, :w]
        img = base + (rng.random((h, w, 3), dtype=np.float32) - 0.5) * 2 * amp[..., None]
    img = np.clip(img, 0, 255).astype(np.uint8)
    if c == 4:
        a = np.full((h, w, 1), 255, np.uint8) if seed % 2 == 0 else rng.integers(0, 256, (h, w, 1), dtype=np.uint8)
        img = np.concatenate([img, a], -1)
    return np.ascontiguousarray(img)


def fast_tol(npx, scale=1.0):
    """Absolute tolerance of a fast-mode value against the reference-order value, in units of the
    compared quantity.  The reference's own value carries the rounding noise of its sequential f32
    sums: up to 0.375 * npx * 2^-24 * (Lmax + |a|max + |b|max [+ alpha]) ~ 1.6e-4 * npx / 4096 in
    raw-metric units (measured: 5e-5 at 64x64), times `scale` = d(value)/d(raw)."""
    return (2.4e-4 * npx / 4096.0 + 1e-5) * max(1.0, abs(scale))


def rel_close(a, b, rel=4e-4, abs_=1e-5):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    bad = np.abs(a - b) > rel * np.abs(b) + abs_
    if bad.any():
        i = int(np.argmax(np.abs(a - b) - rel * np.abs(b)))
        print("rel_close: worst", a[i], b[i], "abs diff", abs(a[i] - b[i]), "allowed", rel * abs(b[i]) + abs_)
    return not bad.any()


def gpu_shrink(ctx, img, bw, bh, metric, factor, filt, flags=0):
    d = ctx.image_upload(img)
    pl = d.shrink(bw, bh, metric, factor, filt, flags)
    descs, pixels = pl.download()
    info = pl.info()
    pl.free()
    d.free()
    return descs, pixels, info


def assert_same_payload(descs, pixels, ref, exact_values, scale=1.0):
    npx = ref.block_width * ref.block_height
    assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"]), "dims"
    assert np.array_equal(descs["offset"], ref.descs["offset"]), "offsets"
    if exact_values:
        assert np.array_equal(descs["value"].view("<u4"), ref.descs["value"].view("<u4")), "stored values bit-exact"
    else:
        assert rel_close(descs["value"], ref.descs["value"], abs_=fast_tol(npx, 1.5 * scale)), "stored values"
    assert pixels.size == ref.payload.size
    assert np.array_equal(pixels, ref.payload), "resampled pixels"


# ---------------------------------------------------------------------------------------------
# analysis
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,bs", [("Big-Ruscher.png", 16), ("Big-Ruscher.png", 32), ("Big-Ruscher.png", 64), ("base.png", 64)])
def test_mad_values_fixture_images(ctx, name, bs):
    img = load_png(name)
    want, _ = O.analyze(img, bs, bs, O.METRIC_OKLAB_MAD, nthreads=8)
    d = ctx.image_upload(img)
    exact, _ = d.analyze(bs, bs, N.METRIC_OKLAB_MAD, N.FLAG_EXACT_VALUES)
    fast, _ = d.analyze(bs, bs, N.METRIC_OKLAB_MAD, 0)
    d.free()
    assert np.array_equal(exact.view("<u4"), want.view("<u4")), "reference-order path must be bit-exact"
    assert rel_close(fast, want, abs_=fast_tol(bs * bs)), float(np.max(np.abs(fast - want)))


@pytest.mark.parametrize("w,h,c,bw,bh", [(257, 131, 3, 32, 32), (260, 132, 4, 64, 64), (259, 130, 4, 64, 64),
                                         (100, 70, 4, 16, 8), (96, 96, 4, 128, 128), (300, 300, 3, 200, 100),
                                         (64, 64, 4, 1, 1), (33, 9, 3, 64, 64), (1, 1, 4, 64, 64), (640, 64, 4, 20, 64)])
def test_mad_values_ragged_shapes(ctx, w, h, c, bw, bh):
    img = synth(w, h, c, seed=w * 7 + h)
    want, _ = O.analyze(img, bw, bh, O.METRIC_OKLAB_MAD, nthreads=8)
    d = ctx.image_upload(img)
    exact, _ = d.analyze(bw, bh, N.METRIC_OKLAB_MAD, N.FLAG_EXACT_VALUES)
    fast, _ = d.analyze(bw, bh, N.METRIC_OKLAB_MAD, 0)
    d.free()
    assert np.array_equal(exact.view("<u4"), want.view("<u4"))
    assert rel_close(fast, want, abs_=fast_tol(bw * bh)), float(np.max(np.abs(fast - want)))


@pytest.mark.parametrize("w,h,c,bw,bh", [(1920, 1080, 3, 32, 32), (258, 131, 3, 32, 32), (260, 132, 4, 64, 64), (99, 70, 4, 16, 8),
                                         (300, 300, 3, 200, 100), (66, 66, 4, 64, 64), (4096, 2115, 4, 64, 64),
                                         (67, 200, 4, 64, 64)])
def test_sobel_values_bit_exact(ctx, w, h, c, bw, bh):
    img = load_png("Big-Ruscher.png") if (w, h) == (1920, 1080) else synth(w, h, c, seed=w + h)
    hz, vr = O.analyze(img, bw, bh, O.METRIC_SOBEL_DIR, nthreads=8)
    d = ctx.image_upload(img)
    ghz, gvr = d.analyze(bw, bh, N.METRIC_SOBEL_DIR)
    d.free()
    assert np.array_equal(ghz.view("<u4"), hz.view("<u4")) and np.array_equal(gvr.view("<u4"), vr.view("<u4"))


def test_sobel_tensor_copy_kernel_matches_shared_memory_kernel(ctx):
    """RGBA + 64x64 tiles take k_analyze_sobel_tma (tiles streamed by tensor copies) when a tensor map can address the rows
    (16-byte aligned base and pitch), and the shared-memory kernel k_analyze_sobel_tile64<4> when they are only 4-byte
    aligned.  Both against the oracle, on a stacked batch too (a tile's box then runs into the next image)."""
    torch = pytest.importorskip("torch")
    imgs = np.stack([synth(323, 150, 4, seed=70 + i) for i in range(3)])
    want = [O.analyze(im, 64, 64, O.METRIC_SOBEL_DIR, nthreads=8) for im in imgs]
    b = ctx.image_upload_batch(imgs)
    ghz, gvr = b.analyze(64, 64, N.METRIC_SOBEL_DIR)
    b.free()
    per = want[0][0].size
    for i, (hz, vr) in enumerate(want):
        assert np.array_equal(ghz.reshape(-1)[i * per:(i + 1) * per].view("<u4"), hz.reshape(-1).view("<u4")), i
        assert np.array_equal(gvr.reshape(-1)[i * per:(i + 1) * per].view("<u4"), vr.reshape(-1).view("<u4")), i
    # the first image once more on each kernel: uploaded (128-byte rows: tensor copies), and wrapped with a base and a pitch
    # that are multiples of 4 but not of 16 (shared memory)
    h, w = imgs[0].shape[:2]
    pitch = w * 4 + 8
    assert pitch % 16 != 0
    host = np.zeros(4 + h * pitch, np.uint8)
    host[4:].reshape(h, pitch)[:, : w * 4] = imgs[0].reshape(h, w * 4)
    buf = torch.from_numpy(host).cuda()
    torch.cuda.synchronize()
    got = []
    for d in (ctx.image_upload(imgs[0]), ctx.image_wrap(buf.data_ptr() + 4, w, h, 4, pitch)):
        got.append(np.stack(d.analyze(64, 64, N.METRIC_SOBEL_DIR)).view("<u4"))
        d.free()
    assert np.array_equal(got[0], got[1])
    assert np.array_equal(got[1], np.stack(want[0]).view("<u4"))


def test_sobel_rejects_blocks_thinner_than_two(ctx):
    d = ctx.image_upload(synth(65, 64, 3, 1))  # trailing column of 1 px: the reference panics
    with pytest.raises(N.PixlzrError):
        d.analyze(64, 64, N.METRIC_SOBEL_DIR)
    d.free()


# ---------------------------------------------------------------------------------------------
# golden files of the reference, through the public API mirror
# ---------------------------------------------------------------------------------------------
def test_golden_big_ruscher_pix_exact_mode():
    """Big-Ruscher.png --from_image(32,32).shrink_by(Lanczos3, 0.125)--> Big-Ruscher.pix, byte for byte."""
    pix = P.Pixlzr.from_image(load_png("Big-Ruscher.png"), 32, 32)
    pix.shrink_by(P.FilterType.Lanczos3, 0.125, exact_values=True)
    assert pix.encode_to_vec() == open(os.path.join(GOLDEN, "Big-Ruscher.pix"), "rb").read()


def test_golden_big_ruscher_pix_fast_mode():
    gold = np.load(os.path.join(GOLDEN, "Big-Ruscher.pix.blocks.npy"))
    pix = P.Pixlzr.from_image(load_png("Big-Ruscher.png"), 32, 32)
    pix.shrink_by(P.FilterType.Lanczos3, 0.125)
    blocks = pix.blocks
    assert [b.width for b in blocks] == gold[:, 1].tolist() and [b.height for b in blocks] == gold[:, 2].tolist()
    vals = np.array([b.block_value for b in blocks], np.float32)
    assert rel_close(vals, gold[:, 0].astype("<u4").view("<f4"), abs_=fast_tol(32 * 32, 1.25 * 1.5))
    ref, _ = O.container_decode(open(os.path.join(GOLDEN, "Big-Ruscher.pix"), "rb").read())
    assert np.array_equal(pix._pixels, ref.payload)


def test_golden_big_ruscher_pix_png():
    """Big-Ruscher.pix --to_image(Nearest)--> Big-Ruscher.pix.png"""
    pix = P.Pixlzr.open(os.path.join(GOLDEN, "Big-Ruscher.pix"))
    assert np.array_equal(pix.to_image(P.FilterType.Nearest), load_png("Big-Ruscher.pix.png"))


@pytest.mark.parametrize("bs", [8, 64])
def test_identity_roundtrip_image_png(bs, tmp_path):
    """main.rs:299-356: image -> pix (file) -> image without shrinking is the identity."""
    img = load_png("image.png")
    pix = P.Pixlzr.from_image(img, bs, bs)
    path = tmp_path / "image.pix"
    pix.save(path)
    back = P.Pixlzr.open(path)
    assert np.array_equal(back.to_image(P.FilterType.Nearest), img)
    assert np.array_equal(back.to_image(P.FilterType.Lanczos3), img)  # full-size blocks: resize is a clone


def test_resize_constant_blocks():
    """block.rs:401-435"""
    for v in (0, 255):
        b = P.PixlzrBlock(np.full((100, 100, 3), v, np.uint8))
        r = b.resize(10, 10, P.FilterType.Lanczos3)
        assert r.dimensions() == (10, 10) and r.block_value is None and (r.data == v).all()


# ---------------------------------------------------------------------------------------------
# shrink / expand against the oracle
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bs", [16, 32, 64])
@pytest.mark.parametrize("down,up", STRATEGIES)
def test_big_ruscher_all_strategies_mad(ctx, bs, down, up):
    img = load_png("Big-Ruscher.png")
    for factor in (1.0, 0.125):
        ref = O.shrink(img, bs, bs, O.METRIC_OKLAB_MAD, factor, down, nthreads=8)
        descs, pixels, info = gpu_shrink(ctx, img, bs, bs, N.METRIC_OKLAB_MAD, factor, down)
        assert_same_payload(descs, pixels, ref, exact_values=False, scale=10 * factor)
        pl = ctx.payload_upload(1920, 1080, bs, bs, 3, descs, pixels)
        out = pl.expand(up)
        pl.free()
        assert np.array_equal(out, O.expand(ref, up, nthreads=8))


@pytest.mark.parametrize("bs", [16, 32, 64])
@pytest.mark.parametrize("down,up", STRATEGIES)
def test_big_ruscher_all_strategies_sobel(ctx, bs, down, up):
    img = load_png("Big-Ruscher.png")
    ref = O.shrink(img, bs, bs, O.METRIC_SOBEL_DIR, 8.0, down, nthreads=8)
    descs, pixels, info = gpu_shrink(ctx, img, bs, bs, N.METRIC_SOBEL_DIR, 8.0, down)
    assert_same_payload(descs, pixels, ref, exact_values=True)
    pl = ctx.payload_upload(1920, 1080, bs, bs, 3, descs, pixels)
    out = pl.expand(up)
    pl.free()
    assert np.array_equal(out, O.expand(ref, up, nthreads=8))


@pytest.mark.parametrize("filt", FILTERS)
def test_base_png_rgba_bench_parameters(ctx, filt):
    """config C1: benches/base.png, 64x64 blocks, shrink_by(filter, 0.25 | 1.0) as benches/bench-00.rs:39,83."""
    img = load_png("base.png")
    for factor in (0.25, 1.0):
        ref = O.shrink(img, 64, 64, O.METRIC_OKLAB_MAD, factor, filt, nthreads=8)
        descs, pixels, info = gpu_shrink(ctx, img, 64, 64, N.METRIC_OKLAB_MAD, factor, filt)
        assert_same_payload(descs, pixels, ref, exact_values=False, scale=10 * factor)
        assert info["bytes"] == ref.payload.size and (info["cols"], info["rows"]) == (17, 26)
    d = ctx.image_upload(img)
    pl = d.shrink(64, 64, N.METRIC_OKLAB_MAD, 1.0, filt, 0)
    out = ctx.image_alloc(1080, 1617, 4)
    pl.expand_to_image(filt, out)  # device-resident encode -> decode, no host round trip
    got = out.download()
    pl.free(); out.free(); d.free()
    assert np.array_equal(got, O.expand(ref, filt, nthreads=8))


@pytest.mark.parametrize("w,h,c,bw,bh", [(257, 131, 3, 32, 32), (260, 132, 4, 64, 64), (259, 130, 4, 64, 48),
                                         (100, 70, 4, 16, 8), (300, 300, 3, 200, 100), (33, 9, 3, 64, 64),
                                         (1, 1, 4, 64, 64), (130, 5, 4, 64, 64), (640, 128, 4, 20, 64)])
@pytest.mark.parametrize("filt", [0, 2, 4])
def test_ragged_shapes_shrink_expand(ctx, w, h, c, bw, bh, filt):
    img = synth(w, h, c, seed=3 * w + h)
    for factor, flags in ((2.0, 0), (0.3, N.FLAG_EXACT_VALUES), (-0.9, 0)):
        ref = O.shrink(img, bw, bh, O.METRIC_OKLAB_MAD, factor, filt, nthreads=8)
        descs, pixels, _ = gpu_shrink(ctx, img, bw, bh, N.METRIC_OKLAB_MAD, factor, filt, flags)
        assert_same_payload(descs, pixels, ref, exact_values=bool(flags), scale=10 * factor)
        pl = ctx.payload_upload(w, h, bw, bh, c, descs, pixels)
        out = pl.expand(filt)
        pl.free()
        assert np.array_equal(out, O.expand(ref, filt, nthreads=8))


def test_expand_arbitrary_block_sizes(ctx):
    """decode side with block sizes no shrink would produce (files written by other tools)."""
    rng = np.random.default_rng(5)
    w, h, bw, bh, c = 150, 100, 64, 64, 4
    cols, rows = O.grid(w, h, bw, bh)
    descs = np.zeros(cols * rows, O.DESC_DTYPE)
    parts, off = [], 0
    for i in range(cols * rows):
        sw, sh = int(rng.integers(1, 70)), int(rng.integers(1, 70))
        descs[i] = (off, 0.5, sw, sh)
        parts.append(rng.integers(0, 256, sw * sh * c, dtype=np.uint8))
        off += sw * sh * c
    payload = np.concatenate(parts)
    ref = O.Shrunk(w, h, bw, bh, c, descs, payload)
    for filt in FILTERS:
        pl = ctx.payload_upload(w, h, bw, bh, c, descs.astype(N.DESC_DTYPE), payload)
        out = pl.expand(filt)
        pl.free()
        assert np.array_equal(out, O.expand(ref, filt, nthreads=8)), filt


def test_process_old_api():
    """process(image, block_size) (process/mod.rs:107-121): Lanczos3 down, Nearest up, RGBA canvas."""
    img = load_png("Big-Ruscher.png")
    out = P.process(img, 32)
    ref = O.shrink(img, 32, 32, O.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, use_factor=False, nthreads=8)
    want = O.expand(ref, O.NEAREST, nthreads=8)
    assert out.shape == (1080, 1920, 4) and (out[..., 3] == 255).all()
    assert np.array_equal(out[..., :3], want)


def test_free_functions():
    img = load_png("Big-Ruscher.png")
    blk = np.ascontiguousarray(img[0:32, 0:32])
    assert np.float32(P.get_block_variance(blk)) == np.float32(O.block_mad(blk))
    hz, vr = P.get_block_variance_directionally(blk)
    ohz, ovr = O.block_sobel(blk)
    assert (np.float32(hz), np.float32(vr)) == (np.float32(ohz), np.float32(ovr))
    blk2 = np.ascontiguousarray(img[320:352, 640:672])
    r = P.reduce_image_section((0.2, 0.4), blk2, P.FilterType.CatmullRom)
    ow, oh, st = O.reduce_dims(0.2, 0.4, 32, 32)
    assert r.dimensions() == (ow, oh) and np.float32(r.block_value) == np.float32(st)
    assert np.array_equal(r.data, O.resize(blk2, ow, oh, O.CATMULLROM))


def test_normalise_global_extension(ctx):
    img = synth(512, 384, 4, seed=11)
    for metric, factor in ((O.METRIC_OKLAB_MAD, 0.05), (O.METRIC_SOBEL_DIR, 1.0)):
        ref = O.shrink(img, 64, 64, metric, factor, O.TRIANGLE, normalise_global=True, nthreads=8)
        descs, pixels, _ = gpu_shrink(ctx, img, 64, 64, metric, factor, O.TRIANGLE, N.FLAG_NORMALISE_GLOBAL | N.FLAG_EXACT_VALUES)
        assert_same_payload(descs, pixels, ref, exact_values=True)
        # without PXZ_FLAG_EXACT_VALUES the Oklab values take the fast path: exact extremes from the tiles that can hold them,
        # reference-order values inside the guard band — dims, offsets and pixels stay bit-exact, stored values within tolerance
        descs, pixels, _ = gpu_shrink(ctx, img, 64, 64, metric, factor, O.TRIANGLE, N.FLAG_NORMALISE_GLOBAL)
        if metric == O.METRIC_SOBEL_DIR:
            assert_same_payload(descs, pixels, ref, exact_values=True)
        else:
            assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"])
            assert np.array_equal(descs["offset"], ref.descs["offset"]) and np.array_equal(pixels, ref.payload)
            assert np.allclose(descs["value"], ref.descs["value"], rtol=2e-3, atol=2e-3 * float(np.max(ref.descs["value"])))


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_normalise_global_fast_path_on_many_levels(ctx, seed):
    """Global normalisation, fast path, on frames with many tiles per level and both extremes shared by several tiles
    (flat tiles): the dims must equal the reference-order run of the same library (PXZ_FLAG_EXACT_VALUES) and the oracle."""
    w, h = 1024, 768
    img = _spread_image(w, h, 4, 64, seed=40 + seed)
    img[0:128, 0:256] = (12, 200, 40, 255)      # flat tiles: several candidates for the minimum
    rng = np.random.default_rng(seed)
    img[640:768, 512:768, :3] = rng.integers(0, 256, (128, 256, 3), dtype=np.uint8)  # white noise: candidates for the maximum
    for factor in (0.02, 0.05, 0.11):
        ref = O.shrink(img, 64, 64, O.METRIC_OKLAB_MAD, factor, O.LANCZOS3, normalise_global=True, nthreads=8)
        fast_d, fast_p, _ = gpu_shrink(ctx, img, 64, 64, O.METRIC_OKLAB_MAD, factor, O.LANCZOS3, N.FLAG_NORMALISE_GLOBAL)
        assert np.array_equal(fast_d["w"], ref.descs["w"]) and np.array_equal(fast_d["h"], ref.descs["h"]), factor
        assert np.array_equal(fast_d["offset"], ref.descs["offset"]) and np.array_equal(fast_p, ref.payload), factor


# ---------------------------------------------------------------------------------------------
# full-size configuration (8K RGBA, 64x64 blocks): size-independent properties + sampled oracle check
# ---------------------------------------------------------------------------------------------
def test_8k_properties(ctx):
    w, h = 7680, 4320
    # white noise: every block keeps its size, so encode -> decode is the identity
    rng = np.random.default_rng(1)
    img = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    d = ctx.image_upload(img)
    pl = d.shrink(64, 64, N.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, 0)
    info = pl.info()
    assert (info["cols"], info["rows"]) == (120, 68) and info["bytes"] == w * h * 4
    descs, pixels = pl.download()
    assert (descs["w"] == 64).all() and set(descs["h"].tolist()) == {64, 32}
    out = ctx.image_alloc(w, h, 4)
    pl.expand_to_image(O.LANCZOS3, out)
    assert np.array_equal(out.download(), img)
    pl.free(); d.free()
    # flat: every block collapses to one pixel of the flat colour
    flat = np.empty((h, w, 4), np.uint8)
    flat[...] = (10, 200, 90, 255)
    d = ctx.image_upload(flat)
    pl = d.shrink(64, 64, N.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, 0)
    descs, pixels = pl.download()
    assert (descs["w"] == 1).all() and (descs["h"] == 1).all() and pixels.size == 120 * 68 * 4
    assert (pixels.reshape(-1, 4) == np.array([10, 200, 90, 255], np.uint8)).all()
    pl.expand_to_image(O.NEAREST, out)
    assert np.array_equal(out.download(), flat)
    pl.free(); d.free(); out.free()


def test_8k_mixed_sampled_against_oracle(ctx):
    w, h = 7680, 4320
    img = synth(w, h, 4, seed=2)
    d = ctx.image_upload(img)
    pl = d.shrink(64, 64, N.METRIC_OKLAB_MAD, 1.0, O.CATMULLROM, 0)
    descs, pixels = pl.download()
    out = ctx.image_alloc(w, h, 4)
    pl.expand_to_image(O.CATMULLROM, out)
    got = out.download()
    pl.free(); out.free(); d.free()
    # offsets are the exclusive scan of the sizes
    sizes = descs["w"].astype(np.uint64) * descs["h"].astype(np.uint64) * 4
    assert np.array_equal(descs["offset"], np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.uint64))
    assert pixels.size == int(sizes.sum())
    assert len(set(descs["w"].tolist())) >= 5  # many levels are populated
    # oracle on a band of block rows (rows 20..23) — same inputs, same block indices
    y0, y1 = 20 * 64, 24 * 64
    ref = O.shrink(np.ascontiguousarray(img[y0:y1]), 64, 64, O.METRIC_OKLAB_MAD, 1.0, O.CATMULLROM, nthreads=8)
    sl = slice(20 * 120, 24 * 120)
    assert np.array_equal(descs["w"][sl], ref.descs["w"]) and np.array_equal(descs["h"][sl], ref.descs["h"])
    assert rel_close(descs["value"][sl], ref.descs["value"], abs_=fast_tol(64 * 64, 15.0))
    o0 = int(descs["offset"][20 * 120])
    assert np.array_equal(pixels[o0:o0 + ref.payload.size], ref.payload)
    assert np.array_equal(got[y0:y1], O.expand(ref, O.CATMULLROM, nthreads=8))


# ---------------------------------------------------------------------------------------------
# opt-in fused-multiply-add resample: dims / offsets / values unchanged, pixels within +-1 LSB
# ---------------------------------------------------------------------------------------------
def psnr(a, b):
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return float("inf") if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


@pytest.mark.parametrize("filt", [1, 2, 3, 4])
def test_fast_resample_within_one_lsb(filt):
    ctx = N.Context(0)
    ctx.set_fast_resample(True)
    for img in (load_png("base.png"), synth(1024, 768, 4, seed=9), synth(1000, 600, 4, seed=8)):
        h, w = img.shape[:2]
        ref = O.shrink(img, 64, 64, O.METRIC_OKLAB_MAD, 1.0, filt, nthreads=8)
        descs, pixels, _ = gpu_shrink(ctx, img, 64, 64, N.METRIC_OKLAB_MAD, 1.0, filt)
        assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"])
        assert np.array_equal(descs["offset"], ref.descs["offset"])
        d = np.abs(pixels.astype(np.int16) - ref.payload.astype(np.int16))
        assert d.max() <= 1, "shrunk pixels must stay within +-1 LSB"
        pl = ctx.payload_upload(w, h, 64, 64, 4, ref.descs.astype(N.DESC_DTYPE), ref.payload)
        out = pl.expand(filt)
        pl.free()
        want = O.expand(ref, filt, nthreads=8)
        d2 = np.abs(out.astype(np.int16) - want.astype(np.int16))
        assert d2.max() <= 1, "expanded pixels must stay within +-1 LSB"
        assert psnr(out, want) > 70.0
        print(f"filter {filt}: shrink differing px {float((d > 0).mean()):.2e}, expand differing px {float((d2 > 0).mean()):.2e}, "
              f"PSNR vs reference decode {psnr(out, want):.1f} dB")
    ctx.close()


# ---------------------------------------------------------------------------------------------
# RGBA fast paths with a NON-opaque alpha channel (the opaque shortcut must not trigger), and mixed images
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("filt", [0, 2, 4])
def test_rgba_fast_path_with_translucent_alpha(ctx, filt):
    img = synth(512, 320, 4, seed=7)  # odd seed: random alpha
    assert img[..., 3].min() < 255
    img[64:192, 128:320, 3] = 255     # a few fully opaque tiles in between: both branches in one launch
    for factor, flags in ((1.0, 0), (0.4, N.FLAG_EXACT_VALUES)):
        ref = O.shrink(img, 64, 64, O.METRIC_OKLAB_MAD, factor, filt, nthreads=8)
        descs, pixels, _ = gpu_shrink(ctx, img, 64, 64, N.METRIC_OKLAB_MAD, factor, filt, flags)
        assert_same_payload(descs, pixels, ref, exact_values=bool(flags), scale=10 * factor)
        pl = ctx.payload_upload(512, 320, 64, 64, 4, descs, pixels)
        out = pl.expand(filt)
        pl.free()
        assert np.array_equal(out, O.expand(ref, filt, nthreads=8))
    want, _ = O.analyze(img, 64, 64, O.METRIC_OKLAB_MAD, nthreads=8)
    d = ctx.image_upload(img)
    fast, _ = d.analyze(64, 64, N.METRIC_OKLAB_MAD, 0)
    exact, _ = d.analyze(64, 64, N.METRIC_OKLAB_MAD, N.FLAG_EXACT_VALUES)
    d.free()
    assert np.array_equal(exact.view("<u4"), want.view("<u4"))
    assert rel_close(fast, want, abs_=fast_tol(64 * 64))


def test_random_shapes_seeded(ctx):
    """Seeded sweep over image / block shapes (trailing blocks of every residue, tiny images, both channel counts)."""
    rng = np.random.default_rng(2024)
    for it in range(24):
        c = int(rng.choice([3, 4]))
        bw, bh = int(rng.choice([8, 16, 24, 32, 64, 96])), int(rng.choice([8, 16, 32, 48, 64, 80]))
        w, h = int(rng.integers(1, 400)), int(rng.integers(1, 300))
        if c == 4 and rng.random() < 0.5:
            w = max(4, w // 4 * 4)  # exercise the aligned RGBA fast paths too
        filt = int(rng.choice(FILTERS))
        factor = float(rng.choice([0.2, 1.0, 3.0]))
        img = synth(w, h, c, seed=it)
        ref = O.shrink(img, bw, bh, O.METRIC_OKLAB_MAD, factor, filt, nthreads=8)
        descs, pixels, _ = gpu_shrink(ctx, img, bw, bh, N.METRIC_OKLAB_MAD, factor, filt)
        assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"]), (it, w, h, c, bw, bh)
        assert np.array_equal(pixels, ref.payload), (it, w, h, c, bw, bh, filt)
        pl = ctx.payload_upload(w, h, bw, bh, c, descs, pixels)
        out = pl.expand(filt)
        pl.free()
        assert np.array_equal(out, O.expand(ref, filt, nthreads=8)), (it, w, h, c, bw, bh, filt)


# ---------------------------------------------------------------------------------------------
# quadtree processing (process/tree.rs) — SURVEY 8f N3
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,bs,thr", [("Big-Ruscher.png", 128, 0.02), ("Big-Ruscher.png", 128, 0.005), ("Big-Ruscher.png", 64, -0.01),
                                         ("base.png", 128, 0.03), ("base.png", 32, 0.01), ("image.png", 256, 0.004)])
def test_tree_process(name, bs, thr):
    img = load_png(name)
    want = O.tree_process(img, thr, bs, bs)
    got = P.tree_process(img, bs, thr)
    assert got.shape == img.shape[:2] + (4,)
    if img.shape[2] == 3:
        assert (got[..., 3] == 255).all()
        got = got[..., :3]
    assert np.array_equal(got, want)
    assert not np.array_equal(got, img)  # something was reduced


def test_tree_process_edge_cases(ctx):
    img = synth(300, 200, 4, seed=5)
    # block size already at the minimum: the input comes back unchanged (tree.rs:35-37)
    assert np.array_equal(P.tree_process(img, 4, 0.01), img)
    # custom filters / minimum block size
    want = O.tree_process(img, 0.02, 64, 32, 8, 8, O.CATMULLROM, O.TRIANGLE)
    got = P.tree_process_custom(img, 0.02, (64, 32), (8, 8), (P.FilterType.CatmullRom, P.FilterType.Triangle))
    assert np.array_equal(got, want)
    # halved sizes that stop being exact are refused, not approximated
    with pytest.raises(N.PixlzrError):
        P.tree_process(img, 100, 0.01)


# ---------------------------------------------------------------------------------------------
# Both resample kernel families stay bit-exact.  By default the library picks by tile count (warp-per-tile from
# 16 tiles per SM — the TMA-fed shrink kernel there — CTA-per-tile below); PXZ_RESAMPLE_KERNELS=warp|cta, read when a
# context is created, forces one.
# ---------------------------------------------------------------------------------------------
def _forced_ctx(kind):
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
def forced_ctx():
    return {"cta": _forced_ctx("cta"), "warp": _forced_ctx("warp")}


@pytest.mark.parametrize("kind", ["warp", "cta"])
@pytest.mark.parametrize("shape,bs,metric,factor,fd,fu", [
    ((520, 776), 64, 0, 1.0, O.LANCZOS3, O.LANCZOS3),      # trailing 8-px / 8-row tiles
    ((300, 420), 32, 0, 1.0, O.CATMULLROM, O.TRIANGLE),
    ((256, 256), 16, 0, 1.0, O.GAUSSIAN, O.NEAREST),
    ((452, 648), 64, 0, 0.5, O.TRIANGLE, O.GAUSSIAN),      # trailing 4 / 8 px: irregular ratios (no slide2 table)
    ((384, 512), 64, 1, 8.0, O.LANCZOS3, O.LANCZOS3),      # Sobel: the two axes get different levels
    ((384, 512), 48, 1, 4.0, O.NEAREST, O.CATMULLROM),
    ((200, 264), 40, 0, 2.0, O.LANCZOS3, O.CATMULLROM),    # 40-px tiles: 40 -> 20 -> 10 -> 5 -> 3 -> 2 -> 1
])
def test_resample_kernel_families_match_oracle(forced_ctx, kind, shape, bs, metric, factor, fd, fu):
    ctx = forced_ctx[kind]
    img = synth(shape[1], shape[0], 4, seed=11)
    img[: shape[0] // 3, : shape[1] // 2, 3] = (img[: shape[0] // 3, : shape[1] // 2, 0] // 2) + 60  # some translucent tiles
    ref = O.shrink(img, bs, bs, metric, factor, fd)
    d = ctx.image_upload(img)
    pl = d.shrink(bs, bs, metric, factor, fd, N.FLAG_EXACT_VALUES)
    descs, px = pl.download()
    assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"])
    assert np.array_equal(descs["offset"], ref.descs["offset"])
    assert np.array_equal(px, ref.payload)
    assert np.array_equal(pl.expand(fu), O.expand(ref, fu))
    # a payload that comes back from the host (pxz_payload_upload builds the work order itself)
    pl2 = ctx.payload_upload(shape[1], shape[0], bs, bs, 4, descs, px)
    assert np.array_equal(pl2.expand(fu), O.expand(ref, fu))
    pl2.free()
    pl.free()
    d.free()


# ---------------------------------------------------------------------------------------------
# RGB images: the input chooses the kernels.  A width that is a multiple of 4, with tiles of at most 64 px on a side and a
# multiple of 4 wide, runs on the RGBA fast kernels (widened with alpha 255, payload narrowed back); any other width runs on
# the 3-channel kernels.  Both must give the oracle's 3-channel result bit for bit, values included.
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,bs,metric,factor,fd,fu", [
    ((200, 264), 64, 0, 1.0, O.LANCZOS3, O.LANCZOS3),  # RGBA kernels
    ((136, 192), 32, 1, 6.0, O.CATMULLROM, O.TRIANGLE),
    ((130, 172), 16, 0, 0.25, O.GAUSSIAN, O.NEAREST),
    ((200, 263), 64, 0, 1.0, O.LANCZOS3, O.LANCZOS3),  # 3-channel kernels
    ((136, 190), 32, 1, 6.0, O.CATMULLROM, O.TRIANGLE),
    ((130, 171), 16, 0, 0.25, O.GAUSSIAN, O.NEAREST),
])
def test_rgb_paths_match_oracle(ctx, shape, bs, metric, factor, fd, fu):
    img = synth(shape[1], shape[0], 3, seed=41)
    ref = O.shrink(img, bs, bs, metric, factor, fd)
    d = ctx.image_upload(img)
    pl = d.shrink(bs, bs, metric, factor, fd, N.FLAG_EXACT_VALUES)
    descs, px = pl.download()
    assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"])
    assert np.array_equal(descs["offset"], ref.descs["offset"])
    assert np.array_equal(descs["value"].view(np.uint32), ref.descs["value"].view(np.uint32))
    assert np.array_equal(px, ref.payload)
    assert np.array_equal(pl.expand(fu), O.expand(ref, fu))
    pl2 = ctx.payload_upload(shape[1], shape[0], bs, bs, 3, descs, px)
    assert np.array_equal(pl2.expand(fu), O.expand(ref, fu))
    pl2.free(); pl.free(); d.free()


# ---------------------------------------------------------------------------------------------
# resize_semantics = fir: the reference's default cargo feature (block.rs:292-333, data_types/mod.rs:65-107).  Integer
# arithmetic: the GPU must equal the oracle's restatement bit for bit (which itself is "parity unpinned" against the crate)
# ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def fir_ctx():
    c = N.Context(0)
    c.set_resize_semantics(N.RESIZE_FIR)
    return c


@pytest.mark.parametrize("shape,ch,bs,metric,factor,fd,fu", [
    ((200, 264), 4, 64, 0, 0.05, O.LANCZOS3, O.LANCZOS3),
    ((200, 264), 4, 64, 0, 0.1, O.TRIANGLE, O.TRIANGLE),      # Hamming down, Bilinear up
    ((136, 192), 4, 32, 1, 6.0, O.CATMULLROM, O.GAUSSIAN),
    ((136, 192), 3, 32, 0, 0.5, O.GAUSSIAN, O.CATMULLROM),
    ((130, 170), 3, 48, 1, 8.0, O.NEAREST, O.LANCZOS3),
    ((96, 128), 4, 16, 0, 2.0, O.LANCZOS3, O.NEAREST),
])
def test_fir_semantics_match_oracle(fir_ctx, shape, ch, bs, metric, factor, fd, fu):
    img = synth(shape[1], shape[0], ch, seed=31)  # odd seed: alpha varies for 4 channels (pre-multiplied path)
    with O.resize_semantics(O.FIR):
        ref = O.shrink(img, bs, bs, metric, factor, fd)
        want = O.expand(ref, fu)
    d = fir_ctx.image_upload(img)
    pl = d.shrink(bs, bs, metric, factor, fd, N.FLAG_EXACT_VALUES)
    descs, px = pl.download()
    assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"])
    assert np.array_equal(px, ref.payload)
    assert np.array_equal(pl.expand(fu), want)
    pl.free(); d.free()
    # the image-crate semantics give other pixels for the same blocks (else this test would prove nothing)
    reduced = (ref.descs["w"].astype(int) * ref.descs["h"] > 1) & ((ref.descs["w"] < bs) | (ref.descs["h"] < bs))
    if fd != O.NEAREST and reduced.sum() > 4:
        assert not np.array_equal(O.shrink(img, bs, bs, metric, factor, fd).payload, ref.payload)


# ---------------------------------------------------------------------------------------------
# batch entry points (pxz_shrink_batch / pxz_expand_batch): one launch per stage over all images, image by image
# identical to the single-image calls — which the other tests hold against the oracle
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["auto", "warp", "cta"])
@pytest.mark.parametrize("shape,bs,metric,factor,fd,fu", [
    ((200, 264), 64, 0, 1.0, O.LANCZOS3, O.LANCZOS3),     # trailing 8-px column, 8-row... per image
    ((136, 192), 32, 1, 6.0, O.CATMULLROM, O.TRIANGLE),   # Sobel: independent axes
])
def test_batch_matches_single_images(forced_ctx, ctx, kind, shape, bs, metric, factor, fd, fu):
    c = ctx if kind == "auto" else forced_ctx[kind]
    h, w = shape
    imgs = np.stack([synth(w, h, 4, seed=20 + i) for i in range(5)])
    batch = c.image_upload_batch(imgs)
    pl = batch.shrink(bs, bs, metric, factor, fd, N.FLAG_EXACT_VALUES)
    info = pl.info()
    assert info["images"] == 5
    descs, px = pl.download()
    per = info["cols"] * info["rows"]
    off = 0
    singles = []
    for i in range(5):
        d = c.image_upload(imgs[i])
        p1 = d.shrink(bs, bs, metric, factor, fd, N.FLAG_EXACT_VALUES)
        d1, x1 = p1.download()
        singles.append(p1.expand(fu))
        p1.free(); d.free()
        db = descs[i * per:(i + 1) * per]
        assert np.array_equal(db["w"], d1["w"]) and np.array_equal(db["h"], d1["h"]), i
        assert np.array_equal(db["value"].view(np.uint32), d1["value"].view(np.uint32)), i
        assert np.array_equal(db["offset"], d1["offset"] + off), i
        assert np.array_equal(px[off:off + x1.size], x1), i
        off += x1.size
    assert off == px.size
    out = pl.expand(fu)
    assert out.shape == imgs.shape
    for i in range(5):
        assert np.array_equal(out[i], singles[i]), i
    # a batch payload that comes back from the host
    pl2 = c.payload_upload_batch(w, h, bs, bs, 4, 5, descs, px)
    assert np.array_equal(pl2.expand(fu), out)
    pl2.free(); pl.free(); batch.free()


# ---------------------------------------------------------------------------------------------
# API gaps closed in round 2: Pixlzr::shrink with the closures the reference passes, and shrink_directionally on blocks
# that already carry a value (pixlzr.rs:124-152, 187-205)
# ---------------------------------------------------------------------------------------------
def test_shrink_with_closures_and_reshrink_of_valued_blocks():
    rng = np.random.default_rng(5)
    img = np.ascontiguousarray(np.concatenate([rng.integers(0, 256, (192, 256, 3), dtype=np.uint8), np.full((192, 256, 1), 255, np.uint8)], -1))
    img[:64, :128, :3] = (img[:64, :128, :3] // 8) + 100  # a few calmer tiles: several levels
    # shrink(filter, |x - avg|, x * k * 10) == shrink_by(filter, k)
    k = 0.5
    a = P.Pixlzr.from_image(img, 64, 64)
    a.shrink(P.FilterType.CatmullRom, lambda x, avg: abs(x - avg), lambda x: x * k * 10.0)
    b = P.Pixlzr.from_image(img, 64, 64)
    b.shrink_by(P.FilterType.CatmullRom, k)
    assert a.encode_to_vec() == b.encode_to_vec()
    # the identity closure is process()'s (process/mod.rs:108-110)
    c = P.Pixlzr.from_image(img, 64, 64)
    c.shrink(P.FilterType.Lanczos3, lambda x, avg: abs(x - avg), lambda x: x)
    ref = O.shrink(img, 64, 64, O.METRIC_OKLAB_MAD, 1.0, O.LANCZOS3, use_factor=False)
    assert np.array_equal(c._descs["w"], ref.descs["w"]) and np.array_equal(c._descs["h"], ref.descs["h"])
    assert np.array_equal(c._pixels, ref.payload)
    # anything else is host-only
    d = P.Pixlzr.from_image(img, 64, 64)
    with pytest.raises(NotImplementedError):
        d.shrink(P.FilterType.Nearest, lambda x, avg: (x - avg) ** 2, lambda x: x)
    # valued blocks: shrink_by skips them, shrink_directionally re-shrinks every block as an image of its own
    pix = P.Pixlzr.decode_from_vec(b.encode_to_vec())
    before = pix.encode_to_vec()
    pix.shrink_by(P.FilterType.Lanczos3, 1.0)
    assert pix.encode_to_vec() == before
    big = [i for i, dsc in enumerate(pix._descs) if dsc["w"] >= 3 and dsc["h"] >= 3]
    if len(big) == len(pix._descs):  # the reference panics on blocks without a 3x3 window (operations.rs:220-221)
        old_descs, old_pixels = pix._descs.copy(), pix._pixels.copy()
        pix.shrink_directionally(P.FilterType.Triangle, 4.0)
        for i, dsc in enumerate(old_descs):
            w, h, o = int(dsc["w"]), int(dsc["h"]), int(dsc["offset"])
            blk = np.ascontiguousarray(old_pixels[o:o + w * h * 4].reshape(h, w, 4))
            r = O.shrink(blk, w, h, O.METRIC_SOBEL_DIR, 4.0, O.TRIANGLE)
            nd = pix._descs[i]
            assert (int(nd["w"]), int(nd["h"])) == (int(r.descs["w"][0]), int(r.descs["h"][0])), i
            no = int(nd["offset"])
            assert np.array_equal(pix._pixels[no:no + r.payload.size], r.payload), i


# ---------------------------------------------------------------------------------------------
# command-line driver (src/bin/main.rs:299-356 and the four conversions)
# ---------------------------------------------------------------------------------------------
def test_cli_conversions(tmp_path):
    from PIL import Image
    src = os.path.join(GOLDEN, "image.png")
    img = load_png("image.png")
    # test_image_to_image: no --force -> identity
    out = str(tmp_path / "test_image.png")
    assert P.cli.main(["-i", src, "-o", out, "-b", "8"]) == 0
    assert np.array_equal(np.array(Image.open(out)), img)
    # test_image_to_pix_to_image
    pix, back = str(tmp_path / "image.pix"), str(tmp_path / "test_image_from_pix.png")
    assert P.cli.main(["-i", src, "-o", pix, "-b", "64"]) == 0
    assert P.cli.main(["-i", pix, "-o", back, "-b", "64"]) == 0
    assert np.array_equal(np.array(Image.open(back)), img)
    # --force shrinks: same bytes as the library calls, and as the oracle
    big = os.path.join(GOLDEN, "Big-Ruscher.png")
    out_pix = str(tmp_path / "big.pix")
    assert P.cli.main(["-i", big, "-o", out_pix, "-b", "32", "-k", "1/8", "-f", "lanczos3", "--force"]) == 0
    ref, _ = O.container_decode(open(os.path.join(GOLDEN, "Big-Ruscher.pix"), "rb").read())
    got, _ = O.container_decode(open(out_pix, "rb").read())
    assert np.array_equal(got.descs["w"], ref.descs["w"]) and np.array_equal(got.descs["h"], ref.descs["h"])
    assert np.array_equal(got.payload, ref.payload)
    # pix -> pix re-tiles the decoded image; pix -> image with another filter
    out_pix2, out_png = str(tmp_path / "re.pixlzr"), str(tmp_path / "big.png")
    assert P.cli.main(["-i", out_pix, "-o", out_pix2, "-b", "64", "-f", "nearest"]) == 0
    assert P.cli.main(["-i", out_pix, "-o", out_png, "-f", "nearest"]) == 0
    assert np.array_equal(np.array(Image.open(out_png)), load_png("Big-Ruscher.pix.png"))
    assert np.array_equal(P.Pixlzr.open(out_pix2).to_image(P.FilterType.Nearest), load_png("Big-Ruscher.pix.png"))
    assert P.cli.main(["-i", str(tmp_path / "missing.png"), "-o", out_png]) == 1


def test_random_shapes_seeded_warp_kernels(forced_ctx):
    """The seeded sweep again, RGBA with 4-px aligned widths and blocks up to 64x64 (what the warp-per-tile kernels take), on a
    context that forces them regardless of the tile count: every shrink runs on the TMA-fed kernel, the tiles without a slide2
    table on k_shrink_warp behind it.  Ragged trailing tiles, odd heights, irregular ratios, Sobel."""
    ctx = forced_ctx["warp"]
    rng = np.random.default_rng(777)
    for it in range(20):
        bw, bh = int(rng.choice([8, 16, 24, 32, 40, 64])), int(rng.choice([8, 16, 24, 32, 48, 64]))
        w, h = max(4, int(rng.integers(4, 420)) // 4 * 4), int(rng.integers(2, 300))
        filt_d, filt_u = int(rng.choice(FILTERS)), int(rng.choice(FILTERS))
        metric = int(rng.choice([O.METRIC_OKLAB_MAD, O.METRIC_OKLAB_MAD, O.METRIC_SOBEL_DIR]))
        if metric == O.METRIC_SOBEL_DIR and (min(bh, h % bh or bh) < 2 or h < 2):
            metric = O.METRIC_OKLAB_MAD
        factor = float(rng.choice([0.2, 1.0, 3.0])) * (8.0 if metric == O.METRIC_SOBEL_DIR else 1.0)
        img = synth(w, h, 4, seed=100 + it)
        if it % 3 == 0:
            img[: h // 2, :, 3] = img[: h // 2, :, 1]  # translucent half
        ref = O.shrink(img, bw, bh, metric, factor, filt_d, nthreads=8)
        descs, pixels, _ = gpu_shrink(ctx, img, bw, bh, metric, factor, filt_d)
        assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"]), (it, w, h, bw, bh, metric)
        assert np.array_equal(pixels, ref.payload), (it, w, h, bw, bh, metric, filt_d)
        pl = ctx.payload_upload(w, h, bw, bh, 4, descs, pixels)
        out = pl.expand(filt_u)
        pl.free()
        assert np.array_equal(out, O.expand(ref, filt_u, nthreads=8)), (it, w, h, bw, bh, metric, filt_u)


def test_sobel_block_without_interior_pixels(ctx):
    """A trailing block 2 rows high has no 3x3 window: the reference's metric is 0/0, the *negative* default NaN on its
    host, which parse_value turns into a 1-pixel block (operations.rs:128-138, 253-254).  Also through the normalise
    extension, whose min/max ignore NaNs."""
    img = synth(136, 50, 4, seed=3)  # 50 = 6 * 8 + 2
    for flags, norm in ((0, False), (N.FLAG_NORMALISE_GLOBAL, True)):
        ref = O.shrink(img, 64, 8, O.METRIC_SOBEL_DIR, 8.0, O.LANCZOS3, normalise_global=norm)
        descs, pixels, _ = gpu_shrink(ctx, img, 64, 8, N.METRIC_SOBEL_DIR, 8.0, O.LANCZOS3, flags)
        assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"])
        assert (descs["w"][-3:] == 1).all() and (descs["h"][-3:] == 1).all()
        assert np.array_equal(pixels, ref.payload)


# ---------------------------------------------------------------------------------------------
# per-block filter pairs (SURVEY.md §8f N4, pxz_ctx_set_strategy): the reference logged which (down, up) pair suits
# each value bucket (strategies.txt) but never used it; the oracle restates the rule on top of the pinned resize.
# ---------------------------------------------------------------------------------------------
def _rainbow_strategy(seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 5, 65).astype(np.uint8), rng.integers(0, 5, 65).astype(np.uint8)


def _spread_image(w, h, c, bs, seed):
    """Noise whose amplitude is log-uniform per block (2^-9 .. 1 of full scale): block values over three decades."""
    rng = np.random.default_rng(seed)
    rows, cols = (h + bs - 1) // bs, (w + bs - 1) // bs
    amp = 128.0 * 2.0 ** (-9.0 * rng.random((rows, cols)))
    amp = np.kron(amp, np.ones((bs, bs)))[:h, :w, None]
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([128 + 60 * np.sin(xx / 97.0), 128 + 60 * np.cos(yy / 131.0), 128 + 40 * np.sin((xx + yy) / 61.0)], -1)
    img = np.clip(base + (rng.random((h, w, 3)) - 0.5) * 2 * amp, 0, 255).astype(np.uint8)
    if c == 4:
        a = np.where(rng.random((h, w, 1)) < 0.5, 255, rng.integers(0, 256, (h, w, 1))).astype(np.uint8)
        a[: h // 2] = 255
        img = np.concatenate([img, a], -1)
    return np.ascontiguousarray(img)


@pytest.mark.parametrize("kind", ["warp", "cta"])
@pytest.mark.parametrize("shape,bs,metric,factor,table", [
    ((520, 776), 64, 0, 0.3, "by_level"),      # trailing 8-px tiles
    ((520, 776), 64, 0, 0.3, "rainbow"),       # every filter in both directions
    ((300, 420), 32, 0, 0.2, "rainbow"),
    ((384, 512), 48, 1, 4.0, "rainbow"),       # Sobel: bucket from hypot(p0, p1) / sqrt(2)
    ((200, 264), 40, 0, 0.1, "by_level"),
    ((97, 131), 16, 0, 0.2, "rainbow"),        # RGB: generic kernels
])
def test_strategy_matches_oracle(forced_ctx, kind, shape, bs, metric, factor, table):
    ctx = forced_ctx[kind]
    channels = 3 if shape == (97, 131) else 4
    img = _spread_image(shape[1], shape[0], channels, bs, seed=5)
    down, up = O.strategy_by_level() if table == "by_level" else _rainbow_strategy(bs + metric)
    ref = O.shrink_strategy(img, bs, bs, metric, factor, down)
    want = O.expand_strategy(ref, up)
    buckets = {O.strategy_bucket(v) for v in ref.descs["value"]}
    assert len(buckets) >= 8 and len({(down[b], up[b]) for b in buckets}) >= 3, "the test image must reach several filter pairs"
    ctx.set_strategy(down, up)
    try:
        d = ctx.image_upload(img)
        pl = d.shrink(bs, bs, metric, factor, O.GAUSSIAN, N.FLAG_EXACT_VALUES)  # the filter argument is ignored
        descs, px = pl.download()
        assert np.array_equal(descs["w"], ref.descs["w"]) and np.array_equal(descs["h"], ref.descs["h"])
        assert np.array_equal(descs["value"].view("<u4"), ref.descs["value"].view("<u4"))
        assert np.array_equal(px, ref.payload)
        assert np.array_equal(pl.expand(O.GAUSSIAN), want)
        # decoder side: descriptors + pixels from the host; the bucket comes from the stored value
        pl2 = ctx.payload_upload(shape[1], shape[0], bs, bs, channels, descs, px)
        assert np.array_equal(pl2.expand(O.TRIANGLE), want)
        pl2.free()
        pl.free()
        d.free()
    finally:
        ctx.set_strategy(None, None)
    # strategy removed: one filter per call again
    ref1 = O.shrink(img, bs, bs, metric, factor, O.CATMULLROM)
    d = ctx.image_upload(img)
    pl = d.shrink(bs, bs, metric, factor, O.CATMULLROM, N.FLAG_EXACT_VALUES)
    assert np.array_equal(pl.download()[1], ref1.payload)
    assert np.array_equal(pl.expand(O.NEAREST), O.expand(ref1, O.NEAREST))
    pl.free()
    d.free()


def test_strategy_uniform_table_equals_plain_filters(ctx):
    """A table with the same pair in every bucket is the ordinary two-filter path."""
    img = synth(400, 300, 4, seed=8)
    ref = O.shrink(img, 32, 32, 0, 0.5, O.CATMULLROM)
    ctx.set_strategy(np.full(65, O.CATMULLROM, np.uint8), np.full(65, O.TRIANGLE, np.uint8))
    try:
        d = ctx.image_upload(img)
        pl = d.shrink(32, 32, 0, 0.5, O.NEAREST, N.FLAG_EXACT_VALUES)
        assert np.array_equal(pl.download()[1], ref.payload)
        assert np.array_equal(pl.expand(O.NEAREST), O.expand(ref, O.TRIANGLE))
        pl.free()
        d.free()
    finally:
        ctx.set_strategy(None, None)
    with pytest.raises(RuntimeError):
        ctx.set_strategy(np.full(65, 7, np.uint8), np.zeros(65, np.uint8))  # unknown filter id


def test_strategy_api_and_container_roundtrip():
    """Pixlzr.shrink_by_strategy -> container -> decode -> to_image_by_strategy, and process_by_strategy."""
    img = load_png(os.path.join(GOLDEN, "Big-Ruscher.png"))
    st = P.Strategy.by_level()
    ref = O.shrink_strategy(img, 32, 32, 0, 0.5, st.down)  # shrink_by: value * factor * 10 is the oracle's default
    want = O.expand_strategy(ref, st.up)
    pix = P.Pixlzr.from_image(img, 32, 32)
    pix.shrink_by_strategy(st, 0.5)
    back = P.Pixlzr.decode_from_vec(pix.encode_to_vec())
    got = back.to_image_by_strategy(st)
    # fast analysis: the guard band also covers the bucket edges where the table changes filters
    assert np.array_equal(got, want)
    assert np.array_equal(back.to_image(P.FilterType.Nearest), O.expand(ref, O.NEAREST))  # and the plain path still works
    ref2 = O.shrink_strategy(img, 64, 64, 0, 1.0, st.down, use_factor=False)
    out = P.process_by_strategy(img, 64)
    want2 = O.expand_strategy(ref2, st.up)
    if want2.shape[2] == 3:
        want2 = np.concatenate([want2, np.full(want2.shape[:2] + (1,), 255, np.uint8)], axis=2)
    assert np.array_equal(out, want2)


# ---------------------------------------------------------------------------------------------
# container stage on the device (SURVEY.md §8f N1, second half): per-block QOI written / read by the GPU,
# byte-identical to the host stage and to the reference's own files
# ---------------------------------------------------------------------------------------------
def test_device_container_reproduces_reference_files(ctx):
    """The committed .pix / .pixlzr fixtures: decoded on the device = decoded on the host; re-encoded on the device =
    the file itself (Big-Ruscher.pix is RGB with a shrunk payload, base.pixlzr RGBA at full size with trailing blocks)."""
    for name in ("Big-Ruscher.pix", "base.pixlzr"):
        with open(os.path.join(GOLDEN, name), "rb") as f:
            data = f.read()
        hdr, descs, pixels = N.container_decode(data)
        pl, filt = ctx.payload_from_container(data)
        d2, p2 = pl.download()
        assert filt == hdr["filter"]
        for k in ("w", "h", "offset"):
            assert np.array_equal(d2[k], descs[k]), (name, k)
        assert np.array_equal(d2["value"].view("<u4"), descs["value"].view("<u4"))
        assert np.array_equal(p2, pixels), name
        assert pl.to_container(max(filt, 0)) == data, name
        assert np.array_equal(pl.expand(O.NEAREST), O.expand(O.Shrunk(hdr["w"], hdr["h"], hdr["bw"], hdr["bh"], hdr["channels"], descs, pixels), O.NEAREST))
        pl.free()


@pytest.mark.parametrize("shape,c,bs,metric,factor", [
    ((300, 420), 4, 32, 0, 0.3),
    ((97, 131), 3, 16, 0, 0.2),
    ((384, 512), 4, 48, 1, 4.0),
    ((64, 64), 4, 64, 0, 1.0),       # one block
    ((250, 333), 3, 40, 0, 0.05),    # mostly tiny blocks
])
def test_device_container_matches_host_stage(ctx, shape, c, bs, metric, factor):
    img = _spread_image(shape[1], shape[0], c, bs, seed=9)
    img[: shape[0] // 2, : shape[1] // 2, :3] = (40, 90, 200)  # flat region: runs, index hits
    d = ctx.image_upload(img)
    pl = d.shrink(bs, bs, metric, factor, O.LANCZOS3, N.FLAG_EXACT_VALUES)
    descs, px = pl.download()
    for vp in (True, False):
        host = N.container_encode(shape[1], shape[0], bs, bs, 4, c, descs, px, None if vp else np.zeros(len(descs), np.uint8))
        dev = pl.to_container(4, vp)
        assert dev == host, "device container differs from the host stage"
    ref = O.shrink(img, bs, bs, metric, factor, O.LANCZOS3)
    assert pl.to_container(4, True) == O.container_encode(ref, 4), "device container differs from the oracle"
    back, filt = ctx.payload_from_container(host)
    d2, p2 = back.download()
    assert filt == 4 and np.array_equal(p2, px) and np.array_equal(d2["w"], descs["w"]) and np.array_equal(d2["h"], descs["h"])
    assert (d2["value"] == 0).all()  # written with values_present = False
    assert np.array_equal(back.expand(O.CATMULLROM), O.expand(ref, O.CATMULLROM))
    back.free()
    pl.free()
    d.free()


def test_device_container_rejects_garbage(ctx):
    with open(os.path.join(GOLDEN, "base.pixlzr"), "rb") as f:
        data = f.read()
    for bad in (b"", b"PIXLZR", data[:100], b"X" + data[1:], data[:-7]):
        with pytest.raises(RuntimeError):
            ctx.payload_from_container(bad)
    pl, _ = ctx.payload_from_container(data)  # the context is still usable afterwards
    pl.free()


def test_device_container_api_equals_three_calls():
    img = load_png("Big-Ruscher.png")
    pix = P.Pixlzr.from_image(img, 32, 32)
    pix.shrink_by(P.FilterType.Lanczos3, 0.125)
    data = pix.encode_to_vec()
    assert P.Pixlzr.encode_image_to_vec(img, 32, 32, P.FilterType.Lanczos3, 0.125) == data
    assert np.array_equal(P.Pixlzr.decode_vec_to_image(data, P.FilterType.CatmullRom),
                          P.Pixlzr.decode_from_vec(data).to_image(P.FilterType.CatmullRom))
    pix = P.Pixlzr.from_image(img, 48, 24)
    pix.shrink_directionally(P.FilterType.Triangle, 2.0)
    assert P.Pixlzr.encode_image_to_vec(img, 48, 24, P.FilterType.Triangle, 2.0, directionally=True) == pix.encode_to_vec()


def test_interleaved_block_row_shards_equal_the_whole_frame(ctx):
    """§8(e), interleaved layout: block row g of the frame on rank g mod N (here 3 ranks, one GPU).  Descriptors, payload,
    the decoded frame and the stitched container file equal the single-GPU result."""
    S = P.sharding
    w, h, bs = 333, 407, 32   # 13 block rows, the last one partial
    img = _spread_image(w, h, 4, bs, seed=22)
    cols, rows = -(-w // bs), -(-h // bs)
    d = ctx.image_upload(img)
    pl = d.shrink(bs, bs, 0, 0.3, O.LANCZOS3, N.FLAG_EXACT_VALUES)
    wd, wp = pl.download()
    whole_file = pl.to_container(4, True)
    whole_out = ctx.image_alloc(w, h, 4)
    pl.expand_to_image(O.LANCZOS3, whole_out)
    whole_px = whole_out.download()
    pl.free(); d.free(); whole_out.free()
    parts, files = [], []
    back = np.zeros_like(img)
    for rank in range(3):
        idx = S.cyclic_block_rows(rows, 3, rank)
        local = S.gather_block_rows(img, bs, idx)
        ds = ctx.image_upload(local)
        ps = ds.shrink(bs, bs, 0, 0.3, O.LANCZOS3, N.FLAG_EXACT_VALUES)
        parts.append(ps.download())
        files.append(ps.to_container(4, True))
        do = ctx.image_alloc(w, local.shape[0], 4)
        ps.expand_to_image(O.LANCZOS3, do)
        S.scatter_block_rows(do.download(), back, bs, idx)
        ps.free(); ds.free(); do.free()
    descs, pixels = S.merge_shards_cyclic(parts, cols)
    nb = cols * rows
    for f in ("w", "h", "offset", "value"):
        assert np.array_equal(descs[f][:nb], wd[f][:nb]), f
    assert pixels.size == wp.size and np.array_equal(pixels, wp)
    assert np.array_equal(back, whole_px)
    assert S.merge_shard_containers_cyclic(files, w, h) == whole_file


def test_device_container_of_block_row_shards_stitches_to_the_whole_file(ctx):
    """§8(e): every rank writes the file of its own block rows on its GPU; the host stitches them (here: 3 shards, one GPU)."""
    S = P.sharding
    w, h, bs = 333, 407, 32   # 13 block rows, the last one partial
    img = _spread_image(w, h, 4, bs, seed=21)
    d = ctx.image_upload(img)
    pl = d.shrink(bs, bs, 0, 0.3, O.LANCZOS3, N.FLAG_EXACT_VALUES)
    whole = pl.to_container(4, True)
    pl.free()
    d.free()
    files = []
    for rank in range(3):
        y0, y1 = S.shard_pixel_rows(h, bs, 3, rank)
        ds = ctx.image_upload(np.ascontiguousarray(img[y0:y1]))
        ps = ds.shrink(bs, bs, 0, 0.3, O.LANCZOS3, N.FLAG_EXACT_VALUES)
        files.append(ps.to_container(4, True))
        ps.free()
        ds.free()
    assert S.merge_shard_containers(files, w, h) == whole
    assert S.merge_shard_containers(files[:2] + [b""] + files[2:], w, h) == whole  # an empty shard is skipped
    with pytest.raises(ValueError):
        S.merge_shard_containers(files[:2], w, h)
