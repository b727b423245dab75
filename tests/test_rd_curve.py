"""Rate-distortion curve on the device (pxz_rd_curve, pxz_shrink_to_error): every point's factor and payload bytes match the
CPU model built from the oracle's block values (test_rd_curve_host.py), every sampled point's error is what pxz_shrink ->
pxz_expand_to_image -> pxz_image_error measures, and the payload of an error budget is pxz_shrink's at the first point within
it."""
import ctypes as C
import os

import numpy as np
import pytest

import pixlzr_b200 as P
from conftest import GOLDEN
from test_rd_curve_host import curve_model
from test_size_target import IMAGES, _same_payload
from test_size_target_host import SizeModel

pytestmark = pytest.mark.gpu
N = P.native
F = P.FilterType
FLAGS = {"plain": 0, "exact": N.FLAG_EXACT_VALUES, "normalise": N.FLAG_NORMALISE_GLOBAL}
METRICS = {"oklab": N.METRIC_OKLAB_MAD, "sobel": N.METRIC_SOBEL_DIR}
# (down, up, resize semantics): one pair per case, cycling
PAIRS = [(F.Lanczos3, F.Lanczos3, N.RESIZE_IMAGE_RS), (F.Nearest, F.Triangle, N.RESIZE_IMAGE_RS),
         (F.CatmullRom, F.Lanczos3, N.RESIZE_FIR), (F.Gaussian, F.Nearest, N.RESIZE_IMAGE_RS)]


@pytest.fixture(scope="module")
def ctxs():
    out = {}
    for sem in (N.RESIZE_IMAGE_RS, N.RESIZE_FIR):
        out[sem] = N.Context(0)
        out[sem].set_resize_semantics(sem)
    return out


def _numpy_sse(a, b):
    return int(((a.astype(np.int64) - b.astype(np.int64)) ** 2).sum())


def _sample(n, count=12):
    return sorted({0, n - 1} | {int(i) for i in np.linspace(0, n - 1, count)})


CASES = [(name, metric, flag) for name in IMAGES for metric in METRICS for flag in FLAGS]


@pytest.mark.parametrize("name,metric,flag", CASES)
def test_curve_points_are_exact(ctxs, name, metric, flag):
    img, bw, bh = IMAGES[name]()
    down, up, sem = PAIRS[CASES.index((name, metric, flag)) % len(PAIRS)]
    ctx = ctxs[sem]
    m, f = METRICS[metric], FLAGS[flag]
    dimg = ctx.image_upload(img)
    try:
        factor, nbytes, sse = dimg.rd_curve(bw, bh, m, int(down), int(up), f)
        model = SizeModel.of_image(img, bw, bh, m, normalise_global=bool(f & N.FLAG_NORMALISE_GLOBAL))
        pats, sizes = curve_model(model)
        assert np.array_equal(factor.view(np.uint32).astype(np.int64), pats)
        assert np.array_equal(nbytes.astype(np.int64), sizes)
        assert len(factor) <= N.rd_curve_bound(img.shape[1], img.shape[0], bw, bh, m)
        for i in _sample(len(factor)):
            pl = dimg.shrink(bw, bh, m, float(factor[i]), int(down), f)
            try:
                assert pl.info()["bytes"] == nbytes[i]
                _, _, total = pl.error(dimg, int(up))
                assert total == sse[i], (i, total, sse[i])
                assert _numpy_sse(pl.expand(int(up)), img) == sse[i]
            finally:
                pl.free()
            if i > 0:  # the pattern below a point gives the point before it: the breakpoint is exact
                below = np.uint32(int(pats[i]) - 1).view(np.float32)
                pb = dimg.shrink(bw, bh, m, float(below), int(down), f)
                assert pb.info()["bytes"] == nbytes[i - 1]
                pb.free()
    finally:
        dimg.free()


def _first_within(sse, budget):
    ok = np.nonzero(sse <= np.uint64(budget))[0]
    return int(ok[0]) if ok.size else None


@pytest.mark.parametrize("name,metric,flag", [("base", "oklab", "plain"), ("synth_rgb", "sobel", "exact"),
                                               ("synth_rgba", "oklab", "normalise"), ("ruscher", "sobel", "plain")])
def test_shrink_to_error(ctxs, name, metric, flag):
    img, bw, bh = IMAGES[name]()
    ctx = ctxs[N.RESIZE_IMAGE_RS]
    m, f = METRICS[metric], FLAGS[flag]
    down, up = int(F.Lanczos3), int(F.Triangle)
    dimg = ctx.image_upload(img)
    try:
        factor, nbytes, sse = dimg.rd_curve(bw, bh, m, down, up, f)
        least = int(sse.min())
        budgets = {least}
        for i in _sample(len(sse), 5):
            budgets |= {int(sse[i]), max(least, int(sse[i]) - 1)}
            if i + 1 < len(sse):
                budgets.add((int(sse[i]) + int(sse[i + 1])) // 2)
        for budget in sorted(budgets):
            j = _first_within(sse, budget)
            pl, k, got_sse = dimg.shrink_to_error(bw, bh, m, budget, down, up, f)
            try:
                assert np.float32(k) == factor[j] and got_sse == sse[j] <= budget
                ref = dimg.shrink(bw, bh, m, k, down, f)
                _same_payload(pl, ref)
                ref.free()
                assert pl.error(dimg, up)[2] == got_sse
                if j > 0:
                    prev = dimg.shrink(bw, bh, m, float(np.nextafter(np.float32(k), np.float32(0))), down, f)
                    assert prev.error(dimg, up)[2] > budget
                    prev.free()
            finally:
                pl.free()
        if least > 0:
            with pytest.raises(N.PixlzrError) as e:
                dimg.shrink_to_error(bw, bh, m, least - 1, down, up, f)
            assert e.value.status == N.E_ARG and str(least) in str(e.value)
    finally:
        dimg.free()


def test_refusals(ctxs):
    img, bw, bh = IMAGES["synth_rgba"]()
    ctx = ctxs[N.RESIZE_IMAGE_RS]
    dimg = ctx.image_upload(img)
    L = N.lib()
    try:
        def status(call):
            with pytest.raises(N.PixlzrError) as e:
                call()
            return e.value.status

        lz = int(F.Lanczos3)
        assert status(lambda: dimg.rd_curve(bw, bh, N.METRIC_OKLAB_MAD, lz, lz, N.FLAG_AFTER_IDENTITY)) == N.E_ARG
        assert status(lambda: dimg.shrink_to_error(bw, bh, N.METRIC_OKLAB_MAD, 10 ** 9, lz, lz, N.FLAG_AFTER_IDENTITY)) == N.E_ARG
        assert status(lambda: dimg.rd_curve(bw, bh, N.METRIC_OKLAB_MAD, 7, lz)) == N.E_ARG
        assert status(lambda: dimg.shrink_to_error(bw, bh, N.METRIC_OKLAB_MAD, 10 ** 9, lz, 9)) == N.E_ARG
        assert status(lambda: dimg.rd_curve(bw, bh, 5, lz, lz)) == N.E_ARG
        sctx = N.Context(0)
        sctx.set_strategy(*N.strategy_by_level())
        simg = sctx.image_upload(img)
        assert status(lambda: simg.rd_curve(bw, bh, N.METRIC_OKLAB_MAD, lz, lz)) == N.E_UNSUPPORTED
        assert status(lambda: simg.shrink_to_error(bw, bh, N.METRIC_OKLAB_MAD, 10 ** 9, lz, lz)) == N.E_UNSUPPORTED
        simg.free()
        batch = ctx.image_upload_batch(np.stack([img, img]))
        assert status(lambda: batch.rd_curve(bw, bh, N.METRIC_OKLAB_MAD, lz, lz)) == N.E_UNSUPPORTED
        assert status(lambda: batch.shrink_to_error(bw, bh, N.METRIC_OKLAB_MAD, 10 ** 9, lz, lz)) == N.E_UNSUPPORTED
        batch.free()
        # cap below the point count: PXZ_E_ARG naming n, *n_out still set, nothing written
        n_full = len(dimg.rd_curve(bw, bh, N.METRIC_SOBEL_DIR, lz, lz)[0])
        fac, nb, se = np.full(1, -1, np.float32), np.zeros(1, np.uint64), np.zeros(1, np.uint64)
        n = C.c_size_t(12345)
        st = L.pxz_rd_curve(ctx.handle, dimg.handle, bw, bh, N.METRIC_SOBEL_DIR, lz, lz, 0, N.ptr(fac), N.ptr(nb), N.ptr(se), 1, C.byref(n))
        assert st == N.E_ARG and n.value == n_full > 1
        assert str(n_full) in L.pxz_last_error(ctx.handle).decode()
        assert fac[0] == -1 and nb[0] == 0 and se[0] == 0
    finally:
        dimg.free()


def test_fused_resample_payload_is_shrinks():
    """With the fused resample arithmetic the error is not claimed exact, but the call succeeds and returns pxz_shrink(k)'s payload."""
    img, bw, bh = IMAGES["base"]()
    ctx = N.Context(0)
    ctx.set_fast_resample(True)
    dimg = ctx.image_upload(img)
    try:
        _, _, sse = dimg.rd_curve(bw, bh, N.METRIC_OKLAB_MAD, int(F.Lanczos3), int(F.Lanczos3))
        budget = int(sse[len(sse) // 2])
        pl, k, _ = dimg.shrink_to_error(bw, bh, N.METRIC_OKLAB_MAD, budget, int(F.Lanczos3), int(F.Lanczos3))
        ref = dimg.shrink(bw, bh, N.METRIC_OKLAB_MAD, k, int(F.Lanczos3))
        _same_payload(pl, ref)
        pl.free()
        ref.free()
    finally:
        dimg.free()


def test_api(ctxs):
    img, bw, bh = IMAGES["base"]()
    rd = P.rd_curve(img, bw, bh, F.Lanczos3, F.Lanczos3, ctx=ctxs[N.RESIZE_IMAGE_RS])
    assert rd.samples == img.size and np.all(np.diff(rd.bytes.astype(np.int64)) > 0)
    target = float(np.median(rd.psnr[np.isfinite(rd.psnr)]))
    pix = P.Pixlzr.from_image(img, bw, bh, ctx=ctxs[N.RESIZE_IMAGE_RS])
    k = pix.shrink_to_psnr(F.Lanczos3, F.Lanczos3, target)
    j = rd.smallest_within(P.sse_budget(target, img.size))
    assert np.float32(k) == rd.factor[j]
    dec = pix.to_image(F.Lanczos3)
    assert P.psnr_of(_numpy_sse(dec, img), img.size) >= target
    with pytest.raises(ValueError):
        pix.shrink_to_psnr(F.Lanczos3, F.Lanczos3, target)  # already shrunk


@pytest.mark.parametrize("out_name", ["out.pix", "out.png"])
def test_cli_target_psnr(tmp_path, capsys, out_name):
    src = os.path.join(GOLDEN, "base.png")
    out = str(tmp_path / out_name)
    assert P.cli.main(["-i", src, "-o", out, "-b", "64", "--target-psnr", "30", "--force", "--psnr"]) == 0
    lines = capsys.readouterr().out.strip().splitlines()
    k = lines[0].split(": ", 1)[1]
    reached = lines[2].split(": ", 1)[1].split(" dB")[0]
    measured = lines[3].split(": ", 1)[1].split(" dB")[0]
    assert lines[1].startswith("payload bytes: ")
    assert float(reached) >= 30.0 and reached == measured
    np.float32(P.parse_shrinking_factor(k))  # -k reads it back
