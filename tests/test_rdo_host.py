"""Rate-distortion optimised encode on the host (no GPU): a model of the per-block hulls and their merge with exact rational
rates, checked on random candidate tables (equal bytes, collinear points, zero and negative gains, single-candidate blocks)
against brute force over every choice of block sizes; the error table of an image built from the oracle's resize; the
curve-length bound; the CLI's --optimal refusals.  The device side is tested in test_rdo.py against this model."""
import itertools
from fractions import Fraction

import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P

N = P.native


def scaled_dim(n: int, level: int) -> int:
    return max(1, -(-n // (1 << level)))


def levels(bw: int, bh: int):
    """(ceil(log2 bw), ceil(log2 bh)): the largest level of each axis; pass of (lx, ly) = lx * (ly_max + 1) + ly"""
    return (bw - 1).bit_length(), (bh - 1).bit_length()


def tile_candidates(tw, th, bw, bh, bpp, sse_of_pass):
    """A block's candidates [(bytes, sse, pass)]: one per distinct dims, at the smallest level pair giving them."""
    lx_max, ly_max = levels(bw, bh)
    seen, out = set(), []
    for lx in range(lx_max + 1):
        for ly in range(ly_max + 1):
            dims = (scaled_dim(tw, lx), scaled_dim(th, ly))
            if dims not in seen:
                seen.add(dims)
                p = lx * (ly_max + 1) + ly
                out.append((dims[0] * dims[1] * bpp, int(sse_of_pass(p)), p))
    return out


def block_hull(cands):
    """Vertices [(bytes, sse, pass)] of a block's hull: by bytes, one per byte count (least sse, then lower pass); from the
    fewest bytes, the points whose sse strictly falls, reduced to their lower convex hull with collinear points kept."""
    best = {}
    for c in cands:
        k = c[0]
        if k not in best or (c[1], c[2]) < (best[k][1], best[k][2]):
            best[k] = c
    pts = [best[k] for k in sorted(best)]
    hull = [pts[0]]
    for p in pts[1:]:
        if p[1] >= hull[-1][1]:
            continue
        # pop the last vertex while it lies strictly above the chord from the one before it to p
        while len(hull) >= 2:
            o, a = hull[-2], hull[-1]
            if (a[1] - o[1]) * (p[0] - o[0]) > (p[1] - o[1]) * (a[0] - o[0]):
                hull.pop()
            else:
                break
        hull.append(p)
    return hull


class Curve:
    """The merged curve of per-block candidate lists: point 0 has every block at its first hull vertex, point j adds the first
    j events by falling rate gain / cost (exact, stable in block then hull order)."""

    def __init__(self, blocks):
        self.hulls = [block_hull(c) for c in blocks]
        events = []
        for b, h in enumerate(self.hulls):
            for k in range(1, len(h)):
                gain, cost = h[k - 1][1] - h[k][1], h[k][0] - h[k - 1][0]
                assert gain > 0 and cost > 0
                events.append((Fraction(gain, cost), b, k, gain, cost))
        events.sort(key=lambda e: -e[0])  # stable
        self.events = events
        b0 = sum(h[0][0] for h in self.hulls)
        s0 = sum(h[0][1] for h in self.hulls)
        self.bytes = np.array([b0] + list(b0 + np.cumsum([e[4] for e in events], dtype=np.int64)), np.int64)
        self.sse = np.array([s0] + list(s0 - np.cumsum([e[3] for e in events], dtype=np.int64)), np.int64)

    def vertex(self, j):
        """per block, the index of its hull vertex at point j"""
        v = [0] * len(self.hulls)
        for _, b, k, _, _ in self.events[:j]:
            assert k == v[b] + 1, "a block's events must come in hull order"
            v[b] = k
        return v

    def passes(self, j):
        return [self.hulls[b][k][2] for b, k in enumerate(self.vertex(j))]

    def best_within(self, max_bytes):
        ok = np.nonzero(self.bytes <= max_bytes)[0]
        return int(ok[-1]) if ok.size else None

    def smallest_within(self, max_sse):
        ok = np.nonzero(self.sse <= max_sse)[0]
        return int(ok[0]) if ok.size else None


def _random_blocks(rng, nblocks, most):
    """candidate lists with repeated byte counts, collinear points, rising and flat errors, single candidates"""
    blocks = []
    for _ in range(nblocks):
        n = int(rng.integers(1, most + 1))
        bytes_ = rng.choice([1, 2, 3, 4, 6, 8, 12, 16], n)
        if rng.random() < 0.3:  # collinear: sse falling linearly in bytes
            sse = [int(100 - 5 * b) for b in bytes_]
        else:
            sse = [int(v) for v in rng.integers(0, 60, n)]
        blocks.append([(int(b), s, p) for p, (b, s) in enumerate(zip(bytes_, sse))])
    return blocks


@pytest.mark.parametrize("seed", range(40))
def test_model_against_brute_force(seed):
    rng = np.random.default_rng(seed)
    blocks = _random_blocks(rng, int(rng.integers(1, 5)), 6)
    c = Curve(blocks)
    assert np.all(np.diff(c.bytes) > 0) and np.all(np.diff(c.sse) < 0)
    distinct = sum(len({b for b, _, _ in cand}) - 1 for cand in blocks)
    assert len(c.bytes) <= 1 + distinct
    # each point's totals are those of its vertices
    for j in range(len(c.bytes)):
        v = c.vertex(j)
        assert sum(c.hulls[b][k][0] for b, k in enumerate(v)) == c.bytes[j]
        assert sum(c.hulls[b][k][1] for b, k in enumerate(v)) == c.sse[j]
    # no choice of candidates has at most a point's bytes and less error
    for choice in itertools.product(*blocks):
        cb, cs = sum(x[0] for x in choice), sum(x[1] for x in choice)
        for j in range(len(c.bytes)):
            assert not (cb <= c.bytes[j] and cs < c.sse[j]), (choice, j)
    # the end: the least error any choice reaches
    assert c.sse[-1] == sum(min(x[1] for x in cand) for cand in blocks)
    # budgets pick the documented points
    for budget in range(0, int(c.bytes[-1]) + 3):
        j = c.best_within(budget)
        assert (j is None) == (budget < c.bytes[0])
        if j is not None:
            assert c.bytes[j] <= budget and (j + 1 == len(c.bytes) or c.bytes[j + 1] > budget)
    for budget in range(int(c.sse[-1]), int(c.sse[0]) + 2):
        j = c.smallest_within(budget)
        assert c.sse[j] <= budget and (j == 0 or c.sse[j - 1] > budget)
    assert c.smallest_within(int(c.sse[-1]) - 1) is None


def test_ties_keep_block_and_hull_order():
    # two blocks with identical hulls: equal rates interleave block by block, each block in hull order
    cand = [(1, 90, 0), (2, 60, 1), (3, 30, 2), (4, 0, 3)]
    c = Curve([cand, cand])
    assert [(e[1], e[2]) for e in c.events] == [(0, 1), (0, 2), (0, 3), (1, 1), (1, 2), (1, 3)]
    # a rate within 1 / (q1 q2) of another, beyond f64 resolution near 2^30
    q1, q2 = 2 ** 20 + 1, 2 ** 20 + 3
    p1, p2 = (2 ** 30) * q1 + 1, (2 ** 30) * q2 + 1
    assert float(Fraction(p1, q1)) == float(Fraction(p2, q2))
    c = Curve([[(1, p2, 0), (1 + q2, 0, 1)], [(1, p1, 0), (1 + q1, 0, 1)]])
    assert [e[1] for e in c.events] == [1, 0]


def test_candidates_of_tiles():
    # a full 64 x 64 tile: 49 pairs, 49 distinct dims, 13 distinct byte counts
    cands = tile_candidates(64, 64, 64, 64, 4, lambda p: 0)
    assert len(cands) == 49 and len({c[0] for c in cands}) == 13
    # a trailing 10-wide tile: levels past 4 repeat width 1, the smallest level pair is kept
    cands = tile_candidates(10, 64, 64, 64, 3, lambda p: p)
    assert len(cands) == 5 * 7
    assert (3, 4 * 7 + 6, 4 * 7 + 6) in cands and all(c[2] // 7 <= 4 for c in cands)


def test_curve_length_bound():
    assert N.rdo_curve_bound(7680, 4320, 64, 64) == 1 + 120 * 68 * 48
    assert N.rdo_curve_bound(203, 98, 32, 16) == 1 + 7 * 7 * (6 * 5 - 1)
    assert N.rdo_curve_bound(5, 5, 1, 1) == 1
    with pytest.raises(ValueError):
        N.rdo_curve_bound(5, 5, 0, 1)


def oracle_table(img, bw, bh, down, up, sem):
    """[passes, blocks] squared error of every block at every level pair: its tile shrunk to the pair's dims with `down` and
    resized back with `up` by the oracle's resize (sem: O.IMAGE_RS or O.FIR), against the tile."""
    resize = O.resize_fir if sem == O.FIR else O.resize
    h, w = img.shape[:2]
    cols, rows = -(-w // bw), -(-h // bh)
    lx_max, ly_max = levels(bw, bh)
    table = np.zeros(((lx_max + 1) * (ly_max + 1), cols * rows), np.int64)
    for r in range(rows):
        for c in range(cols):
            tile = np.ascontiguousarray(img[r * bh:(r + 1) * bh, c * bw:(c + 1) * bw])
            th, tw = tile.shape[:2]
            by_dims = {}
            for lx in range(lx_max + 1):
                for ly in range(ly_max + 1):
                    dims = (scaled_dim(tw, lx), scaled_dim(th, ly))
                    if dims not in by_dims:
                        back = resize(resize(tile, dims[0], dims[1], int(down)), tw, th, int(up))
                        by_dims[dims] = int(((back.astype(np.int64) - tile.astype(np.int64)) ** 2).sum())
                    table[lx * (ly_max + 1) + ly, r * cols + c] = by_dims[dims]
    return table


def oracle_curve(img, bw, bh, down, up, sem):
    """The optimised curve of an image from the oracle table; bytes count the image's channels per pixel."""
    table = oracle_table(img, bw, bh, down, up, sem)
    h, w, ch = img.shape
    cols, rows = -(-w // bw), -(-h // bh)
    blocks = []
    for b in range(cols * rows):
        tw, th = min(bw, w - (b % cols) * bw), min(bh, h - (b // cols) * bh)
        blocks.append(tile_candidates(tw, th, bw, bh, ch, lambda p: table[p, b]))
    return Curve(blocks)


def test_oracle_curve_small():
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (11, 13, 3), dtype=np.uint8)
    c = oracle_curve(img, 8, 4, O.LANCZOS3, O.TRIANGLE, O.IMAGE_RS)
    assert c.bytes[0] == 2 * 3 * 3 and c.sse[-1] == 0
    assert np.all(np.diff(c.bytes) > 0) and np.all(np.diff(c.sse) < 0)
    assert len(c.bytes) <= N.rdo_curve_bound(13, 11, 8, 4)


def test_cli_optimal_refusals(capsys):
    cli = P.cli
    a = cli.parse_args(["-i", "a.png", "-o", "b.pix", "--optimal", "--target-psnr", "40", "--force"])
    assert a.optimal and cli.optimal_error(a) is None
    a = cli.parse_args(["-i", "a.png", "-o", "b.pix", "--optimal", "--payload-bytes", "1000", "--force"])
    assert cli.optimal_error(a) is None
    assert not cli.parse_args(["-i", "a.png", "-o", "b.png"]).optimal
    refused = [
        ["-i", "a.png", "-o", "b.pix", "--optimal", "--force"],                                        # no budget
        ["-i", "a.png", "-o", "b.pix", "--optimal", "--force", "-k", "1/2"],
        ["-i", "a.png", "-o", "b.pix", "--optimal", "--target-psnr", "40", "--force", "-d", "true"],    # a metric
        ["-i", "a.png", "-o", "b.pix", "--optimal", "--payload-bytes", "100", "--force", "-d", "false"],
        ["-i", "a.pix", "-o", "b.png", "--optimal", "--target-psnr", "40", "--force"],                  # container input
        ["-i", "a.png", "-o", "b.pix", "--optimal", "--payload-bytes", "100"],                          # no --force
        ["-i", "a.png", "-o", "b.pix", "--optimal", "--payload-bytes", "100", "--force", "-k", "1"],    # explicit factor
        ["-i", "a.png", "-o", "b.pix", "--optimal", "--payload-bytes", "100", "--target-psnr", "30", "--force"],
    ]
    for argv in refused:
        a = cli.parse_args(argv)
        assert cli.optimal_error(a) or cli.payload_bytes_error(a) or cli.target_psnr_error(a), argv
        with pytest.raises(ValueError):
            cli.run(a)
        assert cli.main(argv) == 2  # refused before any file is opened
    assert "--optimal" in capsys.readouterr().err
