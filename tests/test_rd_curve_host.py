"""Rate-distortion curve on the host (no GPU): a CPU model of the factors at which the payload of pxz_shrink changes, built on
the size model of test_size_target_host.py, checked against scans over the f32 bit patterns; the SSE budget of a PSNR target;
the curve-length bound; the CLI's --target-psnr refusals.  The device side is tested in test_rd_curve.py against this model."""
import numpy as np
import pytest

import pixlzr_b200 as P
from test_size_target_host import MAX_PATTERN, SizeModel, mul_host, parse_values, reduced_dims

N = P.native


def block_dims(model: SizeModel, bits) -> tuple:
    """(w', h') of every block at the factor with bit pattern bits[b] (one pattern per block, or one for all)."""
    k = np.broadcast_to(np.asarray(bits, np.uint32), model.vx.shape).view(np.float32)
    if model.directional:
        v0, v1 = mul_host(model.vx, k), mul_host(model.vy, k)
    else:
        v0 = v1 = mul_host(mul_host(model.vx, k), 10.0)
    return reduced_dims(parse_values(v0), model.tw), reduced_dims(parse_values(v1), model.th)


def block_events(model: SizeModel) -> list:
    """Per block, the sorted bit patterns at which its dims change: for each, the smallest pattern above the last one whose dims
    differ, found by bisection (the dims are monotone in the factor), until the dims of the largest finite factor."""
    nb = model.vx.size
    cur_w, cur_h = block_dims(model, np.ones(nb, np.uint32))
    end_w, end_h = block_dims(model, np.full(nb, MAX_PATTERN, np.uint32))
    p = np.ones(nb, np.int64)
    events = [[] for _ in range(nb)]
    active = (cur_w != end_w) | (cur_h != end_h)
    while active.any():
        lo, hi = p.copy(), np.full(nb, MAX_PATTERN, np.int64)
        while True:
            open_ = active & (hi - lo > 1)
            if not open_.any():
                break
            mid = lo + (hi - lo) // 2
            mw, mh = block_dims(model, mid.astype(np.uint32))
            same = (mw == cur_w) & (mh == cur_h)
            lo = np.where(open_ & same, mid, lo)
            hi = np.where(open_ & ~same, mid, hi)
        nw, nh = block_dims(model, hi.astype(np.uint32))
        for b in np.nonzero(active)[0]:
            events[b].append(int(hi[b]))
        cur_w, cur_h = np.where(active, nw, cur_w), np.where(active, nh, cur_h)
        p = np.where(active, hi, p)
        active = (cur_w != end_w) | (cur_h != end_h)
    return events


def curve_patterns(model: SizeModel) -> np.ndarray:
    """The factors of the curve's points as bit patterns: 1, then every pattern at which some block's dims change."""
    keys = {1}
    for ev in block_events(model):
        keys.update(ev)
    return np.array(sorted(keys), np.int64)


def curve_model(model: SizeModel):
    """(patterns, bytes) of every point of pxz_rd_curve, from the block values alone."""
    pats = curve_patterns(model)
    return pats, np.array([model.size_at(int(b)) for b in pats], np.int64)


def _random_model(seed, directional):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 9))
    special = np.array([0.0, -0.0, np.nan, -np.nan, np.inf, 1e-30, 3.0e-6, 0.5, 17.0], np.float32)

    def values():
        return np.where(rng.random(n) < 0.4, rng.choice(special, n),
                        rng.random(n).astype(np.float32) * 10.0 ** rng.integers(-6, 3, n)).astype(np.float32)

    bw, bh = int(rng.integers(1, 65)), int(rng.integers(1, 65))
    # full tiles and trailing ones (narrower than the block)
    tw = np.where(rng.random(n) < 0.5, bw, rng.integers(1, bw + 1, n))
    th = np.where(rng.random(n) < 0.5, bh, rng.integers(1, bh + 1, n))
    return SizeModel(values(), values(), tw, th, int(rng.choice([3, 4])), directional), bw, bh


@pytest.mark.parametrize("directional", [False, True])
@pytest.mark.parametrize("seed", range(10))
def test_breakpoints_match_a_scan(seed, directional):
    """Every breakpoint is exact (the pattern below it has the previous point's size, every block that changes there had other
    dims one pattern below), and a scan over 2^14 patterns spread over the range finds the size constant between breakpoints."""
    m, bw, bh = _random_model(seed, directional)
    pats, sizes = curve_model(m)
    assert pats[0] == 1 and np.all(np.diff(pats) > 0)
    assert np.all(np.diff(sizes) > 0), "bytes must rise strictly along the curve"
    for i in range(1, len(pats)):
        assert m.size_at(int(pats[i]) - 1) == sizes[i - 1]
    for b, ev in enumerate(block_events(m)):
        for key in ev:
            w1, h1 = block_dims(m, key)
            w0, h0 = block_dims(m, key - 1)
            assert (w1[b], h1[b]) != (w0[b], h0[b])
    scan = np.unique(np.concatenate([np.linspace(1, MAX_PATTERN, 1 << 14).astype(np.int64), pats, pats - 1, [MAX_PATTERN]]))
    scan = scan[scan >= 1]
    point = np.searchsorted(pats, scan, side="right") - 1
    assert all(m.size_at(int(s)) == sizes[i] for s, i in zip(scan, point))


@pytest.mark.parametrize("seed", range(8))
def test_curve_length_bound(seed):
    """A block's dims change at most once per level it steps through: n <= 1 + blocks * (ceil log2 bw + ceil log2 bh), and for
    Oklab-MAD (one level for both axes) 1 + blocks * ceil log2 max(bw, bh)."""
    for directional in (False, True):
        m, bw, bh = _random_model(seed, directional)
        ev = block_events(m)
        lx, ly = (bw - 1).bit_length(), (bh - 1).bit_length()
        per_block = lx + ly if directional else max(lx, ly)
        assert max(len(e) for e in ev) <= per_block
        assert len(curve_patterns(m)) <= 1 + m.vx.size * per_block
    assert N.rd_curve_bound(7680, 4320, 64, 64, N.METRIC_OKLAB_MAD) == 1 + 120 * 68 * 6
    assert N.rd_curve_bound(7680, 4320, 64, 64, N.METRIC_SOBEL_DIR) == 1 + 120 * 68 * 12
    assert N.rd_curve_bound(203, 98, 16, 1, N.METRIC_SOBEL_DIR) == 1 + 13 * 98 * 4


def test_sse_budget_agrees_with_psnr_of():
    """The budget of a target passes it and one more squared error does not, whatever the target."""
    rng = np.random.default_rng(11)
    for _ in range(2000):
        samples = int(rng.integers(1, 1 << 34))
        target = float(rng.uniform(-10.0, 120.0))
        budget = P.sse_budget(target, samples)
        assert P.psnr_of(budget, samples) >= target
        assert P.psnr_of(budget + 1, samples) < target
    # targets that sit exactly on a PSNR some integer SSE gives
    for samples in (3, 12, 7680 * 4320 * 4):
        for sse in (1, 2, 17, 12345):
            target = P.psnr_of(sse, samples)
            assert P.sse_budget(target, samples) == sse
    assert P.sse_budget(float("inf"), 12) == 0
    with pytest.raises(ValueError):
        P.sse_budget(float("nan"), 12)


def test_rate_distortion_smallest_within():
    rd = P.RateDistortion(np.array([1e-45, 0.5, 2.0], np.float32), np.array([10, 20, 40], np.uint64),
                          np.array([900, 300, 310], np.uint64), 100)
    assert rd.smallest_within(310) == 1 and rd.smallest_within(300) == 1 and rd.smallest_within(299) is None
    assert rd.smallest_within(900) == 0
    assert np.allclose(rd.psnr, [P.psnr_of(900, 100), P.psnr_of(300, 100), P.psnr_of(310, 100)])


def test_cli_target_psnr_refusals(capsys):
    cli = P.cli
    a = cli.parse_args(["-i", "a.png", "-o", "b.pix", "--target-psnr", "40", "--force"])
    assert a.target_psnr == 40.0 and cli.target_psnr_error(a) is None
    assert cli.parse_args(["-i", "a.png", "-o", "b.png"]).target_psnr is None
    for bad in ["x", "nan", ""]:
        with pytest.raises(SystemExit):
            cli.parse_args(["-i", "a.png", "-o", "b.pix", "--target-psnr", bad])
    refused = [
        ["-i", "a.pix", "-o", "b.png", "--target-psnr", "40", "--force"],                          # container input
        ["-i", "a.pixlzr", "-o", "b.pix", "--target-psnr", "40", "--force"],
        ["-i", "a.png", "-o", "b.pix", "--target-psnr", "40"],                                     # no --force
        ["-i", "a.png", "-o", "b.pix", "--target-psnr", "40", "--force", "-k", "1"],               # explicit factor
        ["-i", "a.png", "-o", "b.png", "--target-psnr", "40", "--force", "--shrinking-factor=1/2"],
        ["-i", "a.png", "-o", "b.pix", "--target-psnr", "40", "--force", "--payload-bytes", "100"],  # two budgets
        ["-i", "a.png", "-o", "b.png", "--target-psnr", "40", "--force", "--region", "0,0,4,4"],  # region decode
    ]
    for argv in refused:
        a = cli.parse_args(argv)
        assert cli.target_psnr_error(a) or cli.payload_bytes_error(a) or cli.region_error(a), argv
        with pytest.raises(ValueError):
            cli.run(a)
        assert cli.main(argv) == 2  # refused before any file is opened
    assert "--target-psnr" in capsys.readouterr().err
