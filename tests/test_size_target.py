"""Rate control on the device (pxz_shrink_to_size): the chosen factor k is the largest f32 whose pxz_shrink payload fits the
budget, and the payload is byte for byte the one pxz_shrink returns for k.  k is checked bit for bit against a CPU
bisection over the oracle's block values (test_size_target_host.py), the payload against the existing pxz_shrink path."""
import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P
from conftest import load_png
from test_size_target_host import MAX_PATTERN, SizeModel, bisect_factor_bits

pytestmark = pytest.mark.gpu
N = P.native
FLT_MAX = float(np.finfo(np.float32).max)


def synth(w, h, c, seed):
    """smooth base + per-16x16 noise of varying amplitude (many levels); translucent alpha"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.stack([128 + 96 * np.sin(xx / 37.0 + seed), 128 + 96 * np.cos(yy / 41.0), 128 + 64 * np.sin((xx + yy) / 23.0)], -1)
    amp = rng.choice([0, 1, 2, 4, 8, 16, 32, 64, 128], size=((h + 15) // 16, (w + 15) // 16)).astype(np.float32)
    amp = np.kron(amp, np.ones((16, 16), np.float32))[:h, :w]
    img = np.clip(base + (rng.random((h, w, 3), dtype=np.float32) - 0.5) * 2 * amp[..., None], 0, 255).astype(np.uint8)
    if c == 4:
        img = np.concatenate([img, rng.integers(128, 256, (h, w, 1), dtype=np.uint8)], -1)
    return np.ascontiguousarray(img)


# (name, image, bw, bh): RGB on the RGBA kernels, RGBA with a trailing row, RGBA with a trailing column and row, RGB whose
# width is not a multiple of 4 (the 3-channel kernels); every trailing tile is >= 2 px for the directional metric
IMAGES = {
    "ruscher": lambda: (load_png("Big-Ruscher.png"), 32, 32),
    "base": lambda: (load_png("base.png"), 64, 64),
    "synth_rgba": lambda: (synth(203, 150, 4, 1), 32, 32),
    "synth_rgb": lambda: (synth(203, 98, 3, 2), 16, 16),
}
FLAGS = {"plain": 0, "exact": N.FLAG_EXACT_VALUES, "normalise": N.FLAG_NORMALISE_GLOBAL}


@pytest.fixture(scope="module")
def ctx():
    return N.Context(0)


def _budgets(model):
    """about 8 quantiles between the smallest and the full payload, and sizes the payload takes exactly at some factors"""
    lo, hi = model.size_at(1), model.size_at(MAX_PATTERN)
    qs = {int(lo + (hi - lo) * q) for q in np.linspace(0.0, 1.0, 9)}
    steps = {model.size(k) for k in (0.01, 0.1, 0.3, 1.0, 3.0)}
    return sorted(qs | steps | {lo, hi})


def _same_payload(a, b):
    da, pa = a.download()
    db, pb = b.download()
    assert np.array_equal(da.view(np.uint8), db.view(np.uint8)), "descriptors differ"
    assert np.array_equal(pa, pb), "pixels differ"
    assert a.to_container() == b.to_container(), "container bytes differ"


def _check(ctx, img, bw, bh, metric, flags, budget, model=None, filt=int(P.FilterType.Lanczos3)):
    dimg = ctx.image_upload(img)
    try:
        pl, k = dimg.shrink_to_size(bw, bh, metric, budget, filt, flags)
        assert pl.info()["bytes"] <= budget
        ref = dimg.shrink(bw, bh, metric, k, filt, flags)
        _same_payload(pl, ref)
        if k != FLT_MAX:
            up = dimg.shrink(bw, bh, metric, float(np.nextafter(np.float32(k), np.float32(np.inf))), filt, flags)
            assert up.info()["bytes"] > budget
            up.free()
        if model is not None:
            assert np.float32(k).view(np.uint32) == bisect_factor_bits(model, budget), (budget, k)
        pl.free()
        ref.free()
        return k
    finally:
        dimg.free()


@pytest.mark.parametrize("name", sorted(IMAGES))
@pytest.mark.parametrize("metric", [N.METRIC_OKLAB_MAD, N.METRIC_SOBEL_DIR])
@pytest.mark.parametrize("flag", sorted(FLAGS))
def test_factor_is_the_largest_that_fits(ctx, name, metric, flag):
    img, bw, bh = IMAGES[name]()
    model = SizeModel.of_image(img, bw, bh, metric, normalise_global=flag == "normalise")
    for budget in _budgets(model):
        _check(ctx, img, bw, bh, metric, FLAGS[flag], budget, model)


def test_edges_of_the_budget(ctx):
    img, bw, bh = IMAGES["synth_rgba"]()
    model = SizeModel.of_image(img, bw, bh, O.METRIC_OKLAB_MAD)
    smallest = model.size_at(1)
    _check(ctx, img, bw, bh, N.METRIC_OKLAB_MAD, 0, smallest, model)
    dimg = ctx.image_upload(img)
    with pytest.raises(N.PixlzrError) as e:
        dimg.shrink_to_size(bw, bh, N.METRIC_OKLAB_MAD, smallest - 1, int(P.FilterType.Lanczos3))
    assert e.value.status == N.E_ARG and str(smallest) in str(e.value)
    for budget in (img.size, img.size + 1, 1 << 62):
        assert _check(ctx, img, bw, bh, N.METRIC_OKLAB_MAD, 0, budget) == FLT_MAX
    with pytest.raises(N.PixlzrError) as e:
        dimg.shrink_to_size(bw, bh, N.METRIC_OKLAB_MAD, 10000, int(P.FilterType.Lanczos3), N.FLAG_AFTER_IDENTITY)
    assert e.value.status == N.E_ARG
    dimg.free()
    batch = ctx.image_upload_batch(np.stack([img, img]))
    with pytest.raises(N.PixlzrError) as e:
        batch.shrink_to_size(bw, bh, N.METRIC_OKLAB_MAD, 10000, int(P.FilterType.Lanczos3))
    assert e.value.status == N.E_UNSUPPORTED
    batch.free()


def test_two_calls_agree(ctx):
    img, bw, bh = IMAGES["base"]()
    dimg = ctx.image_upload(img)
    budget = SizeModel.of_image(img, bw, bh, O.METRIC_OKLAB_MAD).size(0.5) - 7
    a, ka = dimg.shrink_to_size(bw, bh, N.METRIC_OKLAB_MAD, budget, int(P.FilterType.Lanczos3))
    b, kb = dimg.shrink_to_size(bw, bh, N.METRIC_OKLAB_MAD, budget, int(P.FilterType.Lanczos3))
    assert ka == kb
    _same_payload(a, b)
    dimg.free()


def test_strategy_and_fir_semantics():
    img, bw, bh = IMAGES["synth_rgba"]()
    model = SizeModel.of_image(img, bw, bh, O.METRIC_OKLAB_MAD)
    budgets = [model.size(0.05), model.size(0.5) + 3, (model.size_at(1) + model.size_at(MAX_PATTERN)) // 2]
    sctx = N.Context(0)
    sctx.set_strategy(*N.strategy_by_level())  # per-block filters: no dims change, the factor is the same
    fctx = N.Context(0)
    fctx.set_resize_semantics(N.RESIZE_FIR)
    for c in (sctx, fctx):
        for budget in budgets:
            _check(c, img, bw, bh, N.METRIC_OKLAB_MAD, 0, budget, model)
    rgb, bw, bh = IMAGES["ruscher"]()
    rmodel = SizeModel.of_image(rgb, bw, bh, O.METRIC_SOBEL_DIR)
    _check(fctx, rgb, bw, bh, N.METRIC_SOBEL_DIR, 0, rmodel.size(0.5), rmodel)


def test_api_and_container_counterpart(ctx):
    img, bw, bh = IMAGES["synth_rgba"]()
    budget = SizeModel.of_image(img, bw, bh, O.METRIC_OKLAB_MAD).size(0.2) + 11
    data, k = P.Pixlzr.encode_image_to_vec_sized(img, bw, bh, P.FilterType.Lanczos3, budget, ctx=ctx)
    assert data == P.Pixlzr.encode_image_to_vec(img, bw, bh, P.FilterType.Lanczos3, k, ctx=ctx)
    pix = P.Pixlzr.from_image(img, bw, bh, ctx)
    assert pix.shrink_to_size(P.FilterType.Lanczos3, budget) == k
    ref = P.Pixlzr.from_image(img, bw, bh, ctx)
    ref.shrink_by(P.FilterType.Lanczos3, k)
    assert pix.encode_to_vec() == ref.encode_to_vec() and pix._pixels.size <= budget
    with pytest.raises(ValueError):
        pix.shrink_to_size(P.FilterType.Lanczos3, budget)  # already shrunk: no source image


def test_cli_payload_bytes(tmp_path, capsys):
    from PIL import Image

    img, bw, bh = IMAGES["synth_rgba"]()
    src = str(tmp_path / "in.png")
    Image.fromarray(img).save(src)
    budget = SizeModel.of_image(img, bw, bh, O.METRIC_OKLAB_MAD).size(0.3) + 5
    sized, plain = str(tmp_path / "sized.pix"), str(tmp_path / "plain.pix")
    assert P.cli.main(["-i", src, "-o", sized, "-b", str(bw), "--payload-bytes", str(budget), "--force"]) == 0
    k = capsys.readouterr().out.strip().split()[-1]
    hdr, descs, pixels = N.container_decode(open(sized, "rb").read())
    assert pixels.size <= budget
    assert P.cli.main(["-i", src, "-o", plain, "-b", str(bw), "-k", k, "--force"]) == 0
    assert open(sized, "rb").read() == open(plain, "rb").read()
    out_png = str(tmp_path / "sized.png")
    assert P.cli.main(["-i", src, "-o", out_png, "-b", str(bw), "--payload-bytes", str(budget), "--force"]) == 0
    assert capsys.readouterr().out.strip().split()[-1] == k
