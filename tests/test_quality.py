"""Decode error on the device (pxz_image_error) and the strategy fit built on it (pxz_strategy_measure / pxz_strategy_choose):
exact against numpy and the CPU oracle, identical in the fast and the reference-order Oklab modes, and the fitted table's error
known exactly before encoding."""
import functools
import re

import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P
from conftest import load_png
from test_quality_host import block_error, oracle_measure
from test_size_target import synth

pytestmark = pytest.mark.gpu
N = P.native
NB, NP = N.STRATEGY_BUCKETS, N.FILTER_PAIRS

# (image, bw, bh): RGB on the RGBA kernels, RGBA, RGBA with trailing tiles, RGB whose width is not a multiple of 4 (the
# 3-channel kernels); every trailing tile is >= 2 px for the directional metric
IMAGES = {
    "ruscher": lambda: (load_png("Big-Ruscher.png"), 32, 32),
    "base": lambda: (load_png("base.png"), 64, 64),
    "synth_rgba": lambda: (synth(203, 150, 4, 1), 32, 32),
    "synth_rgb": lambda: (synth(203, 98, 3, 2), 16, 16),
}
FACTOR = {N.METRIC_OKLAB_MAD: 0.2, N.METRIC_SOBEL_DIR: 1.0}  # values spread over many buckets at these factors


@functools.lru_cache(maxsize=None)
def image(name):
    return IMAGES[name]()


@pytest.fixture(scope="module")
def ctx():
    return N.Context(0)


def big_frame():
    """4096 x 2160 RGBA: enough tiles for the library to pick the warp-per-tile resample kernels by itself"""
    return synth(4096, 2160, 4, 7), 32, 32


# ---- 1. pxz_image_error against numpy ------------------------------------------------------------------------------------
@pytest.mark.parametrize("c,w,h,bw,bh", [(4, 203, 150, 32, 32), (3, 203, 98, 16, 16), (4, 200, 120, 24, 10), (3, 96, 64, 7, 13),
                                         (4, 37, 29, 64, 64), (3, 37, 29, 100, 40), (4, 33, 17, 1, 1), (4, 1000, 515, 3, 9)])
def test_image_error_equals_numpy(ctx, c, w, h, bw, bh):
    a = synth(w, h, c, 11)
    b = np.clip(a.astype(np.int16) + np.random.default_rng(w).integers(-40, 41, a.shape), 0, 255).astype(np.uint8)
    b[: h // 3, : w // 2] = a[: h // 3, : w // 2]  # some identical tiles
    da, db = ctx.image_upload(a), ctx.image_upload(b)
    sse, mx, total = da.error(db, bw, bh)
    want_sse, want_max = block_error(a, b, bw, bh)
    assert np.array_equal(sse, want_sse) and np.array_equal(mx, want_max) and total == int(want_sse.sum())
    sse2, mx2, total2 = db.error(da, bw, bh)  # symmetric
    assert np.array_equal(sse2, sse) and np.array_equal(mx2, mx) and total2 == total
    z_sse, z_max, z_total = da.error(da, bw, bh)
    assert z_total == 0 and not z_sse.any() and not z_max.any()
    rep = P.image_error(a, b, bw, bh, ctx)
    assert rep.total_sse == total and rep.psnr == pytest.approx(P.psnr_of(total, a.size))


def test_image_error_on_wrapped_images_with_odd_pitch(ctx):
    torch = pytest.importorskip("torch")
    for c, w, h, pitch, bw, bh in [(4, 203, 77, 203 * 4 + 3, 32, 16), (3, 150, 64, 150 * 3 + 5, 16, 16), (4, 64, 40, 64 * 4 + 8, 16, 8)]:
        a = synth(w, h, c, 3)
        b = np.clip(a.astype(np.int16) + np.random.default_rng(c).integers(-9, 10, a.shape), 0, 255).astype(np.uint8)
        bufs = []
        for shift, x in ((1, a), (0, b)):  # a: rows start one byte past the allocation's alignment as well
            host = np.zeros(shift + h * pitch, np.uint8)
            host[shift:].reshape(h, pitch)[:, : w * c] = x.reshape(h, w * c)
            bufs.append(torch.from_numpy(host).cuda())
        torch.cuda.synchronize()
        wa = ctx.image_wrap(bufs[0].data_ptr() + 1, w, h, c, pitch)
        wb = ctx.image_wrap(bufs[1].data_ptr(), w, h, c, pitch)
        sse, mx, total = wa.error(wb, bw, bh)
        want_sse, want_max = block_error(a, b, bw, bh)
        assert np.array_equal(sse, want_sse) and np.array_equal(mx, want_max) and total == int(want_sse.sum())
        owned = ctx.image_upload(b)  # one wrapped, one owned image
        assert owned.error(wa, bw, bh)[2] == total
        wa.free(), wb.free(), owned.free()


def test_image_error_refusals(ctx):
    a = ctx.image_upload(synth(64, 48, 4, 1))
    for other in (ctx.image_upload(synth(64, 47, 4, 1)), ctx.image_upload(synth(64, 48, 3, 1))):
        with pytest.raises(N.PixlzrError) as e:
            a.error(other, 16, 16)
        assert e.value.status == N.E_ARG
    L = N.lib()
    assert L.pxz_image_error(ctx.handle, a.handle, a.handle, 0, 16, None, None, None) == N.E_ARG
    assert L.pxz_image_error(ctx.handle, a.handle, a.handle, 16, 0, None, None, None) == N.E_ARG
    batch = ctx.image_upload_batch(np.stack([synth(64, 48, 4, 1)] * 2))
    with pytest.raises(N.PixlzrError) as e:
        batch.error(batch, 16, 16)
    assert e.value.status == N.E_UNSUPPORTED
    with pytest.raises(N.PixlzrError) as e:
        batch.strategy_measure(16, 16, N.METRIC_OKLAB_MAD, 0.2)
    assert e.value.status == N.E_UNSUPPORTED
    for x in (a, other, batch):  # see test_measure_leaves_the_installed_strategy
        x.free()


# ---- 2. Payload.error -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(IMAGES))
def test_payload_error_is_the_error_of_the_decode(ctx, name):
    img, bw, bh = image(name)
    src = ctx.image_upload(img)
    pl = src.shrink(bw, bh, N.METRIC_OKLAB_MAD, 0.2, int(P.FilterType.Lanczos3))
    for up in (P.FilterType.Nearest, P.FilterType.CatmullRom):
        got = pl.error(src, int(up))
        dec = pl.expand(int(up))
        want_sse, want_max = block_error(dec, img, bw, bh)
        assert np.array_equal(got[0], want_sse) and np.array_equal(got[1], want_max) and got[2] == int(want_sse.sum())
        assert P.payload_error(pl, img, up).total_sse == got[2]
    # a container round trip decodes to the same pixels
    back, _ = ctx.payload_from_container(pl.to_container())
    assert back.error(src, int(P.FilterType.Nearest))[2] == pl.error(src, int(P.FilterType.Nearest))[2]
    back.free(), pl.free()
    # with a strategy installed: per-block up filters
    sctx = N.Context(0)
    sctx.set_strategy(*N.strategy_by_level())
    ssrc = sctx.image_upload(img)
    spl = ssrc.shrink(bw, bh, N.METRIC_OKLAB_MAD, 0.2, int(P.FilterType.Lanczos3))
    got = spl.error(ssrc, int(P.FilterType.Lanczos3))
    want_sse, _ = block_error(spl.expand(int(P.FilterType.Lanczos3)), img, bw, bh)
    assert np.array_equal(got[0], want_sse)
    spl.free(), ssrc.free(), src.free()


# ---- 3. pxz_strategy_measure against the oracle -----------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def oracle_report(name, metric, use_factor, normalise, fir):
    img, bw, bh = image(name)
    with O.resize_semantics(O.FIR if fir else O.IMAGE_RS):
        return oracle_measure(img, bw, bh, metric, FACTOR[metric], use_factor, normalise)


CASES = [(n, m, f) for n in sorted(IMAGES) for m in (N.METRIC_OKLAB_MAD, N.METRIC_SOBEL_DIR) for f in ("plain", "exact", "normalise")] + \
        [(n, N.METRIC_OKLAB_MAD, "identity") for n in ("synth_rgba", "synth_rgb")]
FLAGS = {"plain": 0, "exact": N.FLAG_EXACT_VALUES, "normalise": N.FLAG_NORMALISE_GLOBAL, "identity": N.FLAG_AFTER_IDENTITY}


@pytest.mark.parametrize("name,metric,flag", CASES)
def test_measure_equals_the_oracle(ctx, name, metric, flag):
    img, bw, bh = image(name)
    dimg = ctx.image_upload(img)
    sse, blocks = dimg.strategy_measure(bw, bh, metric, FACTOR[metric], FLAGS[flag])
    want_sse, want_blocks = oracle_report(name, metric, flag != "identity", flag == "normalise", False)
    assert np.array_equal(blocks, want_blocks)
    assert np.array_equal(sse, want_sse)
    assert int(blocks.sum()) == len(O.shrink(img, bw, bh, metric, FACTOR[metric], 0).descs)
    dimg.free()


@pytest.mark.parametrize("name,metric", [("synth_rgba", N.METRIC_OKLAB_MAD), ("synth_rgb", N.METRIC_OKLAB_MAD),
                                         ("ruscher", N.METRIC_SOBEL_DIR)])
def test_measure_equals_the_oracle_fir(name, metric):
    fctx = N.Context(0)
    fctx.set_resize_semantics(N.RESIZE_FIR)
    img, bw, bh = image(name)
    dimg = fctx.image_upload(img)
    sse, blocks = dimg.strategy_measure(bw, bh, metric, FACTOR[metric], 0)
    want_sse, want_blocks = oracle_report(name, metric, True, False, True)
    assert np.array_equal(blocks, want_blocks) and np.array_equal(sse, want_sse)


# ---- 4. modes agree, calls repeat, the installed strategy stays ------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(IMAGES))
def test_measure_fast_and_exact_oklab_agree(ctx, name):
    img, bw, bh = image(name)
    dimg = ctx.image_upload(img)
    a = dimg.strategy_measure(bw, bh, N.METRIC_OKLAB_MAD, 0.2, 0)
    b = dimg.strategy_measure(bw, bh, N.METRIC_OKLAB_MAD, 0.2, N.FLAG_EXACT_VALUES)
    c = dimg.strategy_measure(bw, bh, N.METRIC_OKLAB_MAD, 0.2, 0)
    for x, y in ((a, b), (a, c)):
        assert np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1])
    dimg.free()


def test_measure_leaves_the_installed_strategy(ctx):
    img, bw, bh = image("synth_rgba")
    table = (np.random.default_rng(1).integers(0, 5, NB).astype(np.uint8), np.random.default_rng(2).integers(0, 5, NB).astype(np.uint8))

    def decode(c):
        d = c.image_upload(img)
        pl = d.shrink(bw, bh, N.METRIC_OKLAB_MAD, 0.2, int(P.FilterType.Lanczos3))
        return pl.download()[1], pl.expand(int(P.FilterType.Lanczos3))

    sctx = N.Context(0)
    sctx.set_strategy(*table)
    before = decode(sctx)
    sctx.image_upload(img).strategy_measure(bw, bh, N.METRIC_OKLAB_MAD, 0.2)
    after = decode(sctx)
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])
    # and the strategy does not leak into the measure: the same report as on a context without one
    a = sctx.image_upload(img).strategy_measure(bw, bh, N.METRIC_OKLAB_MAD, 0.2)
    b = ctx.image_upload(img).strategy_measure(bw, bh, N.METRIC_OKLAB_MAD, 0.2)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    # an error on the way out (Sobel on a 1-px trailing column) still restores the table
    bad = sctx.image_upload(synth(65, 64, 4, 1))
    with pytest.raises(N.PixlzrError) as e:
        bad.strategy_measure(16, 16, N.METRIC_SOBEL_DIR, 1.0)
    assert e.value.status == N.E_ARG
    again = decode(sctx)
    assert np.array_equal(before[1], again[1])
    # the traceback in `e` keeps this frame alive: free the image now, so that no later garbage collection finalises it
    # after its context
    bad.free()


# ---- 5. the fitted table's error is known before encoding -------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(IMAGES) + ["big"])
def test_fitted_table_error_is_predicted_exactly(ctx, name):
    img, bw, bh = big_frame() if name == "big" else image(name)
    factor = FACTOR[N.METRIC_OKLAB_MAD]
    fit, rep = P.Strategy.fit([img], bw, bh, factor, ctx=ctx)
    sctx = N.Context(0)
    sctx.set_strategy(fit.down, fit.up)
    src = sctx.image_upload(img)
    pl = src.shrink(bw, bh, N.METRIC_OKLAB_MAD, factor, int(P.FilterType.Lanczos3))
    got = pl.error(src, int(P.FilterType.Lanczos3))[2]
    assert got == rep.total(fit)
    for d in range(5):
        for u in range(5):
            assert got <= rep.total(P.Strategy.uniform(d, u))
    assert got <= rep.total(P.Strategy.by_level())
    # blocks[] is the histogram of the buckets of the reference-order stored values
    ex = ctx.image_upload(img).shrink(bw, bh, N.METRIC_OKLAB_MAD, factor, 0, N.FLAG_EXACT_VALUES)
    values = ex.download()[0]["value"]
    hist = np.bincount([N.strategy_bucket(v) for v in values], minlength=NB)
    assert np.array_equal(rep.blocks, hist)
    pl.free(), src.free(), ex.free()


def test_fit_sums_reports_over_images(ctx):
    imgs = [synth(203, 150, 4, 1), synth(203, 150, 4, 5)]
    fit, rep = P.Strategy.fit(imgs, 32, 32, 0.2, ctx=ctx)
    parts = [ctx.image_upload(i).strategy_measure(32, 32, N.METRIC_OKLAB_MAD, 0.2) for i in imgs]
    assert np.array_equal(rep.sse, parts[0][0] + parts[1][0]) and np.array_equal(rep.blocks, parts[0][1] + parts[1][1])
    down, up = N.strategy_choose(rep.sse, rep.blocks)
    assert np.array_equal(fit.down, down) and np.array_equal(fit.up, up)


# ---- 6. the CLI's --psnr ----------------------------------------------------------------------------------------------------
def _printed(out):
    m = re.search(r"psnr: (\S+) dB, max error: (\d+)", out)
    assert m, out
    return float(m.group(1)), int(m.group(2))


def test_cli_psnr(tmp_path, capsys):
    from PIL import Image

    img, bw, bh = image("synth_rgba")
    src = str(tmp_path / "in.png")
    Image.fromarray(img).save(src)
    cases = [(["-o", str(tmp_path / "a.pix"), "-k", "1/4", "--force", "-f", "catmull-rom"], "pix"),
             (["-o", str(tmp_path / "b.png"), "-k", "1/4", "--force"], "image"),
             (["-o", str(tmp_path / "c.pix"), "--payload-bytes", str(img.size // 5), "--force"], "pix"),
             (["-o", str(tmp_path / "d.png"), "--payload-bytes", str(img.size // 5), "--force", "-f", "triangle"], "image"),
             (["-o", str(tmp_path / "e.pix")], "pix")]
    for extra, kind in cases:
        assert P.cli.main(["-i", src, "-b", str(bw)] + extra + ["--psnr"]) == 0
        psnr, mx = _printed(capsys.readouterr().out)
        out = extra[1]
        filt = P.cli.FILTERS[extra[extra.index("-f") + 1]] if "-f" in extra else P.FilterType.Lanczos3
        if kind == "pix":
            dec = P.Pixlzr.decode_vec_to_image(open(out, "rb").read(), filt)
        else:
            dec = np.array(Image.open(out))
        d = dec.astype(np.int64) - img.astype(np.int64)
        sse = int((d * d).sum())
        want = P.psnr_of(sse, img.size)
        assert (psnr == want == float("inf")) or abs(psnr - want) < 1e-5
        assert mx == int(np.abs(d).max())
