"""Rate control on the host (no GPU): a vectorised CPU model of the payload size as a function of the shrinking factor, the
bisection over f32 bit patterns that pxz_shrink_to_size must agree with, and the CLI's --payload-bytes refusals.  The
device side is tested in test_size_target.py against this model."""
import functools

import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P

N = P.native
MAX_PATTERN = 0x7F7FFFFF  # FLT_MAX: patterns 1 .. MAX_PATTERN are the finite factors > 0


@functools.lru_cache(maxsize=1)
def level_thresholds() -> np.ndarray:
    """thr[k] = smallest f32 p > 0 with the oracle's level exponent >= -k (operations.rs:147-148), k = 0..40: the exponent is
    monotone in p, so a bisection over bit patterns with the oracle's scalar rule finds each edge."""
    thr = np.zeros(41, np.float32)
    for k in range(41):
        lo, hi = 0, 0x7F800000  # level_exp(lo) < -k (0: none known), level_exp(hi) >= -k (+inf)
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if O.level_exp(float(np.uint32(mid).view(np.float32))) >= -k:
                hi = mid
            else:
                lo = mid
        thr[k] = np.uint32(hi).view(np.float32)
    return thr


def parse_values(v: np.ndarray) -> np.ndarray:
    """parse_value (operations.rs:128-138), vectorised: negative values (NaN with the sign bit too) -> max(1 + v, 0)."""
    v = np.asarray(v, np.float32)
    with np.errstate(invalid="ignore"):
        one = np.float32(1) + v
        neg = np.where(one > 0, one, np.float32(0))
    return np.where(np.signbit(v), neg, v).astype(np.float32)


def reduced_dims(p: np.ndarray, n: np.ndarray) -> np.ndarray:
    """(n * level).max(1).ceil() (operations.rs:150-151) for parsed values p and tile sides n: level = 2^-k with k the number
    of thresholds above p (NaN and +inf: k = 0; 0 and below thr[40]: one pixel for every side the format allows)."""
    with np.errstate(invalid="ignore"):
        k = (p[:, None] < level_thresholds()[None, :]).sum(1).astype(np.int64)
    n = np.asarray(n, np.int64)
    return np.maximum(1, (n + (np.int64(1) << k) - 1) >> k)


def mul_host(a: np.ndarray, b) -> np.ndarray:
    """a * b in f32 as the reference's host computes it: a NaN operand comes back unchanged, sign included."""
    a = np.asarray(a, np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        return np.where(np.isnan(a), a, a * np.float32(b)).astype(np.float32)


def normalise(v: np.ndarray) -> np.ndarray:
    """PXZ_FLAG_NORMALISE_GLOBAL: (v - min) / (max - min) over the non-NaN values, 0 for an empty range (NaNs stay)."""
    v = np.asarray(v, np.float32)
    ok = v[~np.isnan(v)]
    if ok.size == 0:
        return np.zeros_like(v)
    mn, mx = ok.min(), ok.max()
    rg = np.float32(mx - mn)
    if not rg > 0:
        return np.zeros_like(v)
    with np.errstate(invalid="ignore"):
        return np.where(np.isnan(v), v, (v - mn) / rg).astype(np.float32)


class SizeModel:
    """Payload bytes of pxz_shrink(k) from raw block values (oracle.analyze): x * k * 10 for Oklab-MAD (pixlzr.rs:162),
    (hz * k, vr * k) for the directional metric (pixlzr.rs:199), then parse_value -> level -> dims."""

    def __init__(self, vx, vy, tw, th, channels, directional, normalise_global=False):
        vx, vy = np.asarray(vx, np.float32), np.asarray(vy, np.float32)
        if normalise_global:
            vx, vy = normalise(vx), normalise(vy)
        self.vx, self.vy = vx, (vy if directional else vx)
        self.tw, self.th = np.asarray(tw, np.int64), np.asarray(th, np.int64)
        self.channels, self.directional = channels, directional

    @classmethod
    def of_image(cls, img, bw, bh, metric, normalise_global=False):
        H, W, c = img.shape
        vx, vy = O.analyze(np.ascontiguousarray(img), bw, bh, metric)
        cols, rows = O.grid(W, H, bw, bh)
        tw = np.minimum(bw, W - np.arange(cols) * bw)
        th = np.minimum(bh, H - np.arange(rows) * bh)
        return cls(vx, vy, np.tile(tw, rows), np.repeat(th, cols), c, metric == O.METRIC_SOBEL_DIR, normalise_global)

    def size(self, k) -> int:
        k = np.float32(k)
        if self.directional:
            v0, v1 = mul_host(self.vx, k), mul_host(self.vy, k)
        else:
            v0 = v1 = mul_host(mul_host(self.vx, k), 10.0)
        w = reduced_dims(parse_values(v0), self.tw)
        h = reduced_dims(parse_values(v1), self.th)
        return int((w * h).sum()) * self.channels

    def size_at(self, bits: int) -> int:
        return self.size(np.uint32(bits).view(np.float32))


def bisect_factor_bits(model: SizeModel, max_bytes: int) -> int:
    """Bit pattern of the largest finite f32 k > 0 with model.size(k) <= max_bytes (0: not even the smallest factor fits)."""
    lo, hi = 0, MAX_PATTERN + 1
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if model.size_at(mid) <= max_bytes:
            lo = mid
        else:
            hi = mid
    return lo


def _random_model(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 9))
    special = np.array([0.0, -0.0, np.nan, -np.nan, np.inf, 1e-30, 3.0e-6, 0.5, 17.0], np.float32)
    vx = np.where(rng.random(n) < 0.4, rng.choice(special, n), rng.random(n).astype(np.float32) * 10.0 ** rng.integers(-6, 3, n))
    vy = np.where(rng.random(n) < 0.4, rng.choice(special, n), rng.random(n).astype(np.float32) * 10.0 ** rng.integers(-6, 3, n))
    tw, th = rng.integers(1, 17, n), rng.integers(1, 17, n)
    return SizeModel(vx.astype(np.float32), vy.astype(np.float32), tw, th, int(rng.choice([3, 4])), bool(seed % 2))


def test_vectorised_dims_follow_the_oracle():
    """The vectorised value -> dims rule is the oracle's scalar reduce_dims, NaN of both signs and zeros included."""
    rng = np.random.default_rng(3)
    v = np.concatenate([np.array([0.0, -0.0, np.nan, -np.nan, np.inf, -np.inf, -0.5, -1.0, -2.0, 1.0], np.float32),
                        (rng.random(300) * 10.0 ** rng.integers(-13, 2, 300)).astype(np.float32),
                        level_thresholds(), np.nextafter(level_thresholds(), np.float32(0))])
    n = rng.integers(1, 65536, v.size)
    got = reduced_dims(parse_values(v), n)
    want = np.array([O.reduce_dims(float(x), float(x), int(m), int(m))[0] for x, m in zip(v, n)])
    assert np.array_equal(got, want)


@pytest.mark.parametrize("seed", range(12))
def test_bisection_matches_a_scan(seed):
    """On small random value sets the bisection's factor fits, its successor does not, and a scan over 2^15 patterns spread
    over the whole range finds no fitting factor above it: the size is monotone in the factor, so it is the largest one."""
    m = _random_model(seed)
    scan = np.unique(np.concatenate([np.linspace(1, MAX_PATTERN, 1 << 15).astype(np.int64), [1, MAX_PATTERN]]))
    sizes = np.array([m.size_at(int(b)) for b in scan])
    assert np.all(np.diff(sizes) >= 0), "size not monotone in the factor"
    for budget in sorted({int(sizes[0]) - 1, int(sizes[0]), int(sizes[-1]), int(sizes[len(sizes) // 3]),
                          int(sizes[len(sizes) // 3]) + 1, int(np.median(sizes)), int(sizes[-1]) + 5}):
        bits = bisect_factor_bits(m, budget)
        if bits == 0:
            assert m.size_at(1) > budget
            continue
        assert m.size_at(bits) <= budget
        assert bits == MAX_PATTERN or m.size_at(bits + 1) > budget
        assert bits >= scan[sizes <= budget].max()


def test_format_shrinking_factor_reads_back():
    rng = np.random.default_rng(5)
    ks = np.concatenate([rng.integers(1, MAX_PATTERN, 20000, dtype=np.uint32), [1, 2, MAX_PATTERN, 0x3F800000]]).astype(np.uint32)
    for k in ks.view(np.float32):
        assert np.float32(P.parse_shrinking_factor(P.api.format_shrinking_factor(k))) == k


def test_cli_payload_bytes_refusals(tmp_path, capsys):
    cli = P.cli
    a = cli.parse_args(["-i", "a.png", "-o", "b.pix", "--payload-bytes", "1000", "--force"])
    assert a.payload_bytes == 1000 and cli.payload_bytes_error(a) is None
    assert cli.parse_args(["-i", "a.png", "-o", "b.pix"]).payload_bytes is None
    for bad in ["-1", "x", "1.5"]:
        with pytest.raises(SystemExit):
            cli.parse_args(["-i", "a.png", "-o", "b.pix", "--payload-bytes", bad])
    refused = [
        ["-i", "a.pix", "-o", "b.png", "--payload-bytes", "10", "--force"],        # container input
        ["-i", "a.pixlzr", "-o", "b.pix", "--payload-bytes", "10", "--force"],
        ["-i", "a.png", "-o", "b.pix", "--payload-bytes", "10"],                   # no --force
        ["-i", "a.png", "-o", "b.pix", "--payload-bytes", "10", "--force", "-k", "1"],  # explicit factor
        ["-i", "a.png", "-o", "b.png", "--payload-bytes", "10", "--force", "--shrinking-factor=1/2"],
    ]
    for argv in refused:
        a = cli.parse_args(argv)
        assert cli.payload_bytes_error(a), argv
        with pytest.raises(ValueError):
            cli.run(a)
        assert cli.main(argv) == 2  # refused before any file is opened
    assert "--payload-bytes" in capsys.readouterr().err
