"""Rate-distortion optimised encode on the device (pxz_rdo_curve, pxz_rdo_shrink_to_size / _to_error): the curve equals the
CPU model built from the oracle's per-block error table (test_rdo_host.py); the payload of a budget has the point's bytes, its
decode the point's error, every block the descriptor of its level pair, and every reader decodes it; the curve is never above
the factor curves of either metric."""
import os

import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P
from conftest import GOLDEN, load_png
from test_rdo_host import levels, oracle_curve
from test_size_target import IMAGES, synth

pytestmark = pytest.mark.gpu
N = P.native
F = P.FilterType
# (down, up, resize semantics): one pair per case, cycling
PAIRS = [(F.Lanczos3, F.Lanczos3, N.RESIZE_IMAGE_RS), (F.Nearest, F.Triangle, N.RESIZE_IMAGE_RS),
         (F.CatmullRom, F.Lanczos3, N.RESIZE_FIR), (F.Gaussian, F.Nearest, N.RESIZE_IMAGE_RS)]
# the images of the factor budgets, and non-square blocks with trailing tiles on both axes
CASES = dict(IMAGES, wide_blocks=lambda: (synth(203, 150, 4, 5), 32, 16))
ORACLE_SEM = {N.RESIZE_IMAGE_RS: O.IMAGE_RS, N.RESIZE_FIR: O.FIR}


@pytest.fixture(scope="module")
def ctxs():
    out = {}
    for sem in (N.RESIZE_IMAGE_RS, N.RESIZE_FIR):
        out[sem] = N.Context(0)
        out[sem].set_resize_semantics(sem)
    return out


def _numpy_sse(a, b):
    return int(((a.astype(np.int64) - b.astype(np.int64)) ** 2).sum())


def _sample(n, count=6):
    return sorted({0, n - 1} | {int(i) for i in np.linspace(0, n - 1, count)})


def _expected_descs(img, bw, bh, passes):
    """(w, h, value) of every block at its level pair: pxz_reduce_dims(2^-lx, 2^-ly, tw, th)"""
    h, w = img.shape[:2]
    cols = -(-w // bw)
    _, ly_max = levels(bw, bh)
    out = []
    for b, p in enumerate(passes):
        lx, ly = divmod(p, ly_max + 1)
        tw, th = min(bw, w - (b % cols) * bw), min(bh, h - (b // cols) * bh)
        out.append(N.reduce_dims(2.0 ** -lx, 2.0 ** -ly, tw, th))
    return out


def _check_payload(ctx, dimg, img, bw, bh, pl, up, sem, want_bytes, want_sse, passes):
    assert pl.info()["bytes"] == want_bytes
    assert pl.error(dimg, int(up))[2] == want_sse
    dec = pl.expand(int(up))
    assert _numpy_sse(dec, img) == want_sse
    descs, _ = pl.download()
    exp = _expected_descs(img, bw, bh, passes)
    assert np.array_equal(descs["w"], [e[0] for e in exp]) and np.array_equal(descs["h"], [e[1] for e in exp])
    assert np.array_equal(descs["value"], np.array([e[2] for e in exp], np.float32))
    # readers: the device container reader, and the host one expanded by the oracle
    data = pl.to_container(0, True)
    back, _ = ctx.payload_from_container(data)
    try:
        assert np.array_equal(back.expand(int(up)), dec)
    finally:
        back.free()
    hdr, hdescs, hpixels = N.container_decode(data)
    with O.resize_semantics(ORACLE_SEM[sem]):
        ref = O.expand(O.Shrunk(hdr["w"], hdr["h"], hdr["bw"], hdr["bh"], hdr["channels"], hdescs, hpixels), int(up))
    assert np.array_equal(ref, dec)


@pytest.mark.parametrize("name", list(CASES))
def test_curve_and_payloads_are_exact(ctxs, name):
    img, bw, bh = CASES[name]()
    down, up, sem = PAIRS[list(CASES).index(name) % len(PAIRS)]
    ctx = ctxs[sem]
    model = oracle_curve(img, bw, bh, down, up, ORACLE_SEM[sem])
    dimg = ctx.image_upload(img)
    try:
        nbytes, sse = dimg.rdo_curve(bw, bh, int(down), int(up))
        assert np.array_equal(nbytes.astype(np.int64), model.bytes)
        assert np.array_equal(sse.astype(np.int64), model.sse)
        assert len(nbytes) <= N.rdo_curve_bound(img.shape[1], img.shape[0], bw, bh) and sse[-1] == 0
        for j in _sample(len(nbytes)):
            for call, budget in (("rdo_shrink_to_size", int(nbytes[j])), ("rdo_shrink_to_error", int(sse[j]))):
                pl, got_bytes, got_sse = getattr(dimg, call)(bw, bh, budget, int(down), int(up))
                try:
                    assert (got_bytes, got_sse) == (nbytes[j], sse[j]), (call, j)
                    _check_payload(ctx, dimg, img, bw, bh, pl, up, sem, int(nbytes[j]), int(sse[j]), model.passes(j))
                finally:
                    pl.free()
        # a budget between two points picks the one the rule names
        j = len(nbytes) // 2
        pl, got_bytes, _ = dimg.rdo_shrink_to_size(bw, bh, int(nbytes[j + 1]) - 1, int(down), int(up))
        assert got_bytes == nbytes[j]
        pl.free()
        pl, got_bytes, got_sse = dimg.rdo_shrink_to_error(bw, bh, int(sse[j - 1]) - 1, int(down), int(up))
        assert (got_bytes, got_sse) == (nbytes[j], sse[j])
        pl.free()
    finally:
        dimg.free()


@pytest.mark.parametrize("name", list(IMAGES))
def test_dominates_the_factor_curves(ctxs, name):
    img, bw, bh = IMAGES[name]()
    down, up = int(F.Lanczos3), int(F.Triangle)
    dimg = ctxs[N.RESIZE_IMAGE_RS].image_upload(img)
    try:
        rb, rs = dimg.rdo_curve(bw, bh, down, up)
        for metric in (N.METRIC_OKLAB_MAD, N.METRIC_SOBEL_DIR):
            _, fb, fs = dimg.rd_curve(bw, bh, metric, down, up)
            # the first optimised point with bytes >= B (past the end: the last point, with sse 0 and fewer bytes)
            j = np.minimum(np.searchsorted(rb, fb, side="left"), len(rb) - 1)
            assert np.all(rs[j] <= fs), metric
            for i in _sample(len(fs), 4):
                pa, _, _ = dimg.shrink_to_error(bw, bh, metric, int(fs[i]), down, up)
                b_a = pa.info()["bytes"]
                pa.free()
                po, got_bytes, got_sse = dimg.rdo_shrink_to_error(bw, bh, int(fs[i]), down, up)
                po.free()
                assert got_sse <= fs[i] and got_bytes <= rb[min(np.searchsorted(rb, b_a, side="left"), len(rb) - 1)]
    finally:
        dimg.free()


def test_refusals(ctxs):
    img, bw, bh = IMAGES["synth_rgba"]()
    ctx = ctxs[N.RESIZE_IMAGE_RS]
    lz = int(F.Lanczos3)
    dimg = ctx.image_upload(img)

    def status(call):
        with pytest.raises(N.PixlzrError) as e:
            call()
        return e.value.status

    try:
        assert status(lambda: dimg.rdo_curve(bw, bh, 7, lz)) == N.E_ARG
        assert status(lambda: dimg.rdo_shrink_to_error(bw, bh, 10 ** 9, lz, 9)) == N.E_ARG
        assert status(lambda: dimg.rdo_shrink_to_size(0, bh, 10 ** 9, lz, lz)) == N.E_ARG
        nbytes, _ = dimg.rdo_curve(bw, bh, lz, lz)
        with pytest.raises(N.PixlzrError) as e:
            dimg.rdo_shrink_to_size(bw, bh, int(nbytes[0]) - 1, lz, lz)
        assert e.value.status == N.E_ARG and str(int(nbytes[0])) in str(e.value)
        pl, got, _ = dimg.rdo_shrink_to_size(bw, bh, int(nbytes[0]), lz, lz)
        assert got == nbytes[0]
        pl.free()
        sctx = N.Context(0)
        sctx.set_strategy(*N.strategy_by_level())
        simg = sctx.image_upload(img)
        assert status(lambda: simg.rdo_curve(bw, bh, lz, lz)) == N.E_UNSUPPORTED
        assert status(lambda: simg.rdo_shrink_to_error(bw, bh, 10 ** 9, lz, lz)) == N.E_UNSUPPORTED
        simg.free()
        batch = ctx.image_upload_batch(np.stack([img, img]))
        assert status(lambda: batch.rdo_curve(bw, bh, lz, lz)) == N.E_UNSUPPORTED
        assert status(lambda: batch.rdo_shrink_to_size(bw, bh, 10 ** 9, lz, lz)) == N.E_UNSUPPORTED
        batch.free()
    finally:
        dimg.free()


def test_api(ctxs):
    img, bw, bh = IMAGES["synth_rgba"]()
    ctx = ctxs[N.RESIZE_IMAGE_RS]
    curve = P.rdo_curve(img, bw, bh, F.Lanczos3, F.Lanczos3, ctx=ctx)
    assert curve.samples == img.size and np.all(np.diff(curve.bytes.astype(np.int64)) > 0)
    budget = int(curve.bytes[len(curve.bytes) // 3])
    pix = P.Pixlzr.from_image(img, bw, bh, ctx=ctx)
    got_bytes, got_sse = pix.shrink_optimally_to_size(F.Lanczos3, F.Lanczos3, budget)
    j = curve.best_within(budget)
    assert (got_bytes, got_sse) == (curve.bytes[j], curve.sse[j])
    assert _numpy_sse(pix.to_image(F.Lanczos3), img) == got_sse
    with pytest.raises(ValueError):
        pix.shrink_optimally_to_size(F.Lanczos3, F.Lanczos3, budget)  # already shrunk
    target = float(np.median(curve.psnr[np.isfinite(curve.psnr)]))
    pix = P.Pixlzr.from_image(img, bw, bh, ctx=ctx)
    got_bytes, got_sse = pix.shrink_optimally_to_psnr(F.Lanczos3, F.Lanczos3, target)
    j = curve.smallest_within(P.sse_budget(target, img.size))
    assert (got_bytes, got_sse) == (curve.bytes[j], curve.sse[j])
    assert P.psnr_of(_numpy_sse(pix.to_image(F.Lanczos3), img), img.size) >= target


def test_cli_optimal(tmp_path, capsys):
    src = os.path.join(GOLDEN, "base.png")
    source = load_png("base.png")
    out, dec = str(tmp_path / "out.pix"), str(tmp_path / "dec.png")
    assert P.cli.main(["-i", src, "-o", out, "-b", "64", "--optimal", "--target-psnr", "35", "--force"]) == 0
    lines = capsys.readouterr().out.strip().splitlines()
    assert lines[0].startswith("payload bytes: ")
    reached = lines[1].split(": ", 1)[1].split(" dB")[0]
    assert float(reached) >= 35.0
    assert P.cli.main(["-i", out, "-o", dec, "-f", "lanczos3"]) == 0
    from PIL import Image
    decoded = np.array(Image.open(dec))
    assert P.cli.format_psnr(P.psnr_of(_numpy_sse(decoded, source), source.size)) == reached
    budget = int(lines[0].split(": ", 1)[1]) // 2
    assert P.cli.main(["-i", src, "-o", str(tmp_path / "small.png"), "-b", "64", "--optimal", "--payload-bytes", str(budget),
                       "--force"]) == 0
    lines = capsys.readouterr().out.strip().splitlines()
    assert int(lines[0].split(": ", 1)[1]) <= budget
