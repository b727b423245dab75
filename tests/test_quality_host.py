"""Decode error and strategy fit, host side: the table choice (pxz_strategy_choose), the decomposition of a strategy decode's
error into per-pair block errors that the device fit relies on (checked on the CPU oracle alone), the PSNR formula and the
CLI's --psnr refusals.  No GPU needed."""
import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P

N = P.native
NB, NP = N.STRATEGY_BUCKETS, N.FILTER_PAIRS


def block_error(a, b, bw, bh):
    """numpy restatement of pxz_image_error: (sse uint64 [rows, cols], max uint8 [rows, cols]) over the tiles of (bw, bh)."""
    assert a.shape == b.shape
    h, w, _ = a.shape
    d = np.abs(a.astype(np.int64) - b.astype(np.int64))
    rows, cols = -(-h // bh), -(-w // bw)
    # zero padding up to whole tiles adds nothing to either figure
    d = np.pad(d, ((0, rows * bh - h), (0, cols * bw - w), (0, 0))).reshape(rows, bh, cols, bw, -1)
    sse = (d * d).sum(axis=(1, 3, 4)).astype(np.uint64)
    mx = d.max(axis=(1, 3, 4)).astype(np.uint8)
    return sse, mx


def synth(w, h, c, seed):
    """smooth base + per-8x8 noise of varying amplitude (values in many buckets)"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    base = np.stack([128 + 96 * np.sin(xx / 17.0 + seed), 128 + 96 * np.cos(yy / 19.0), 128 + 64 * np.sin((xx + yy) / 11.0)], -1)
    amp = rng.choice([0, 1, 2, 4, 8, 16, 32, 64, 128], size=((h + 7) // 8, (w + 7) // 8)).astype(np.float32)
    amp = np.kron(amp, np.ones((8, 8), np.float32))[:h, :w]
    img = np.clip(base + (rng.random((h, w, 3), dtype=np.float32) - 0.5) * 2 * amp[..., None], 0, 255).astype(np.uint8)
    if c == 4:
        img = np.concatenate([img, rng.integers(128, 256, (h, w, 1), dtype=np.uint8)], -1)
    return np.ascontiguousarray(img)


def oracle_measure(img, bw, bh, metric, factor, use_factor=True, normalise=False, nthreads=0):
    """The report pxz_strategy_measure returns, from the oracle: per down filter one shrink, per up filter one expand, numpy
    block errors added per pxo_strategy_bucket of the oracle's stored values."""
    import os
    nthreads = nthreads or os.cpu_count() or 1
    sse = np.zeros((NB, NP), np.uint64)
    blocks = np.zeros(NB, np.uint32)
    h, w, _ = img.shape
    for down in range(5):
        s = O.shrink(img, bw, bh, metric, factor, down, use_factor, normalise, nthreads)
        bk = np.array([O.strategy_bucket(v) for v in s.descs["value"]], np.int64)
        if down == 0:
            blocks = np.bincount(bk, minlength=NB).astype(np.uint32)
        for up in range(5):
            e, _ = block_error(O.expand(s, up, nthreads), img, bw, bh)
            np.add.at(sse[:, down * 5 + up], bk, e.reshape(-1))
    return sse, blocks


# ---- pxz_strategy_choose ---------------------------------------------------------------------------------------------------
def test_choose_takes_the_argmin_per_bucket():
    rng = np.random.default_rng(3)
    sse = rng.integers(0, 1 << 40, (NB, NP)).astype(np.uint64)
    blocks = rng.integers(1, 100, NB).astype(np.uint32)
    down, up = N.strategy_choose(sse, blocks)
    best = sse.argmin(axis=1)  # random 40-bit sums: no ties
    assert np.array_equal(down.astype(np.int64) * 5 + up, best)


def test_choose_ties_and_empty_buckets():
    bd, bu = N.strategy_by_level()
    base_pair = bd.astype(np.int64) * 5 + bu
    sse = np.full((NB, NP), 100, np.uint64)
    blocks = np.ones(NB, np.uint32)
    # bucket 0: base's pair among the least -> kept; bucket 1: a tie without base's pair -> lowest index;
    # bucket 2: empty bucket with a better pair -> base's pair; bucket 3: one clear winner
    sse[0, base_pair[0]] = 5
    sse[0, 17] = 5
    sse[1, [9, 21]] = 7
    sse[2, 3] = 1
    blocks[2] = 0
    sse[3, 12] = 0
    down, up = N.strategy_choose(sse, blocks)
    pair = down.astype(np.int64) * 5 + up
    assert pair[0] == base_pair[0]
    assert pair[1] == 9
    assert pair[2] == base_pair[2]
    assert pair[3] == 12
    # all equal: every bucket keeps base's pair; base None means by_level
    flat = np.zeros((NB, NP), np.uint64)
    assert np.array_equal(np.stack(N.strategy_choose(flat, blocks)), np.stack((bd, bu)))
    other = (np.full(NB, 2, np.uint8), np.full(NB, 3, np.uint8))
    assert np.array_equal(np.stack(N.strategy_choose(flat, blocks, other)), np.stack(other))
    assert np.array_equal(np.stack(N.strategy_choose(sse, np.zeros(NB, np.uint32), other)), np.stack(other))


def test_choose_refuses_null_arguments_and_unknown_filters():
    sse = np.zeros((NB, NP), np.uint64)
    blocks = np.ones(NB, np.uint32)
    out = np.zeros(2 * NB, np.uint8)
    L = N.lib()
    assert L.pxz_strategy_choose(None, N.ptr(blocks), None, N.ptr(out)) == N.E_ARG
    assert L.pxz_strategy_choose(N.ptr(sse), None, None, N.ptr(out)) == N.E_ARG
    assert L.pxz_strategy_choose(N.ptr(sse), N.ptr(blocks), None, None) == N.E_ARG
    with pytest.raises(N.PixlzrError):
        N.strategy_choose(sse, blocks, (np.full(NB, 5, np.uint8), np.zeros(NB, np.uint8)))


def test_report_totals():
    rng = np.random.default_rng(5)
    sse = rng.integers(0, 1 << 30, (NB, NP)).astype(np.uint64)
    rep = P.StrategyReport(sse, np.ones(NB, np.uint32))
    s = P.Strategy.by_level()
    assert rep.total(s) == sum(int(sse[b, int(s.down[b]) * 5 + int(s.up[b])]) for b in range(NB))
    assert rep.total(P.Strategy.uniform(P.FilterType.Gaussian, P.FilterType.Triangle)) == int(sse[:, 3 * 5 + 1].sum())


# ---- the decomposition the fit relies on (oracle only) --------------------------------------------------------------------
@pytest.mark.parametrize("c,w,h,bw,bh,metric,factor", [(4, 75, 61, 16, 16, O.METRIC_OKLAB_MAD, 0.2),
                                                        (3, 70, 45, 12, 8, O.METRIC_OKLAB_MAD, 0.2),
                                                        (4, 75, 61, 16, 16, O.METRIC_SOBEL_DIR, 1.0)])
def test_strategy_error_is_the_sum_of_per_pair_block_errors(c, w, h, bw, bh, metric, factor):
    img = synth(w, h, c, seed=w + c)
    # per-pair block errors from uniform oracle runs; the stored values do not depend on the filter
    per_pair = {}
    values = None
    for down in range(5):
        s = O.shrink(img, bw, bh, metric, factor, down)
        if values is None:
            values = s.descs["value"].copy()
        assert np.array_equal(s.descs["value"], values) and np.array_equal(s.descs["w"], O.shrink(img, bw, bh, metric, factor, 0).descs["w"])
        for up in range(5):
            per_pair[down * 5 + up] = block_error(O.expand(s, up), img, bw, bh)[0].reshape(-1)
    bk = np.array([O.strategy_bucket(v) for v in values])
    assert len(set(bk.tolist())) > 3, "the image should spread over several buckets"
    rng = np.random.default_rng(11)
    for _ in range(3):
        down_lut = rng.integers(0, 5, NB).astype(np.uint8)
        up_lut = rng.integers(0, 5, NB).astype(np.uint8)
        s = O.shrink_strategy(img, bw, bh, metric, factor, down_lut)
        out = O.expand_strategy(s, up_lut)
        got = int(block_error(out, img, bw, bh)[0].sum())
        want = sum(int(per_pair[int(down_lut[k]) * 5 + int(up_lut[k])][i]) for i, k in enumerate(bk))
        assert got == want


def test_numpy_block_error_on_trailing_tiles():
    a = synth(13, 9, 3, 1)
    b = a.copy()
    b[8, 12, 2] ^= 0x0F  # last pixel, in the trailing tile of both axes
    sse, mx = block_error(a, b, 4, 4)
    assert sse.shape == (3, 4) and int(sse.sum()) == int(mx[2, 3]) ** 2 and int(mx[2, 3]) == abs(int(a[8, 12, 2]) - int(b[8, 12, 2]))


# ---- PSNR and the CLI ------------------------------------------------------------------------------------------------------
def test_psnr_formula():
    assert P.psnr_of(0, 100) == float("inf")
    assert P.psnr_of(255 * 255 * 12, 12) == pytest.approx(0.0)
    assert P.psnr_of(12, 12) == pytest.approx(20 * np.log10(255.0))
    rep = P.ErrorReport(np.array([[3, 5]], np.uint64), np.array([[1, 2]], np.uint8), 8, 4 * 2 * 3)
    assert rep.mse == pytest.approx(8 / 24) and rep.psnr == pytest.approx(10 * np.log10(255.0 ** 2 / (8 / 24)))
    assert rep.max_error == 2
    assert P.cli.format_psnr(float("inf")) == "inf" and P.cli.format_psnr(31.25) == "31.250000"


@pytest.mark.parametrize("src,dst", [("in.pix", "out.png"), ("in.pixlzr", "out.pix"), ("in.PIX", "out")])
def test_cli_refuses_psnr_for_container_inputs(tmp_path, capsys, src, dst):
    rc = P.cli.main(["-i", str(tmp_path / src), "-o", str(tmp_path / dst), "--psnr"])
    assert rc == 2
    assert "--psnr" in capsys.readouterr().err
    assert not (tmp_path / dst).exists()


def test_cli_psnr_accepts_image_inputs():
    for argv in (["-i", "a.png", "-o", "b.pix", "--psnr"], ["-i", "a.png", "-o", "b.png", "--psnr", "--force"],
                 ["-i", "a.png", "-o", "b.pix", "--psnr", "--force", "--payload-bytes", "100"]):
        args = P.cli.parse_args(argv)
        assert args.psnr and P.cli.psnr_error(args) is None
    assert P.cli.parse_args(["-i", "a.png", "-o", "b.pix"]).psnr is False
