"""Random access on the host (no GPU): cropping a .pxlzr file to a block window without decoding it, the header-only
read, and the CLI's --region.  The device side (windows of payloads, pixel rectangles) is tested in test_region.py."""
import os
import struct

import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P
from conftest import GOLDEN

N = P.native


def _windows(cols, rows):
    """(c0, r0, nc, nr): a single block, a full row, a full column, the trailing corner, the whole grid, and some more"""
    wins = {(0, 0, 1, 1), (0, rows // 2, cols, 1), (cols // 2, 0, 1, rows), (cols - 1, rows - 1, 1, 1), (0, 0, cols, rows),
            (cols - 2, 0, 2, rows), (0, rows - 2, cols, 2), (1, 1, cols - 2, rows - 2)}
    rng = np.random.default_rng(7)
    for _ in range(12):
        c0, r0 = int(rng.integers(0, cols)), int(rng.integers(0, rows))
        wins.add((c0, r0, int(rng.integers(1, cols - c0 + 1)), int(rng.integers(1, rows - r0 + 1))))
    return sorted(wins)


@pytest.mark.parametrize("c", [3, 4])
def test_crop_equals_the_file_of_the_cropped_image(c):
    """The crop of an oracle-written file is byte for byte the file the oracle writes for the block-aligned crop of the
    image: a block's record depends only on that block, and the window keeps the trailing-tile rule."""
    rng = np.random.default_rng(11 + c)
    w, h, bs = 150, 210, 32  # 5 x 7 blocks, trailing column (22 px) and row (18 px)
    img = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
    img[40:120, 10:90] = 77  # flat area: blocks of several levels
    img[:, 100:] //= 8
    whole = O.container_encode(O.shrink(img, bs, bs, O.METRIC_OKLAB_MAD, 0.02, O.LANCZOS3), 4)
    cols, rows = O.grid(w, h, bs, bs)
    for (c0, r0, nc, nr) in _windows(cols, rows):
        x0, y0, x1, y1 = c0 * bs, r0 * bs, min(w, (c0 + nc) * bs), min(h, (r0 + nr) * bs)
        want = O.container_encode(O.shrink(np.ascontiguousarray(img[y0:y1, x0:x1]), bs, bs, O.METRIC_OKLAB_MAD, 0.02, O.LANCZOS3), 4)
        assert N.container_crop(whole, c0, r0, nc, nr) == want, (c0, r0, nc, nr)
    assert N.container_crop(whole, 0, 0, cols, rows) == whole
    # any buffer: a memoryview (an mmap behaves the same) gives the same bytes
    assert N.container_crop(memoryview(whole), 1, 2, 3, 4) == N.container_crop(whole, 1, 2, 3, 4)


@pytest.mark.parametrize("name", ["Big-Ruscher.pix", "base.pixlzr"])
def test_header_and_crop_of_reference_files(name):
    raw = open(os.path.join(GOLDEN, name), "rb").read()
    hdr, descs, pixels = N.container_decode(raw)
    head = N.container_header(raw)
    assert head == {k: hdr[k] for k in ("w", "h", "bw", "bh", "filter")}
    cols, rows = N.grid(hdr["w"], hdr["h"], hdr["bw"], hdr["bh"])
    c = hdr["channels"]
    # the crop decodes to the window's blocks: same descriptors (offsets re-packed) and pixels
    for (c0, r0, nc, nr) in [(0, 0, 1, 1), (cols - 1, rows - 1, 1, 1), (2, 3, 5, 4), (0, 0, cols, rows)]:
        sub = N.container_crop(raw, c0, r0, nc, nr)
        shdr, sdescs, spx = N.container_decode(sub)
        assert (shdr["w"], shdr["h"]) == (min(hdr["w"], (c0 + nc) * hdr["bw"]) - c0 * hdr["bw"],
                                         min(hdr["h"], (r0 + nr) * hdr["bh"]) - r0 * hdr["bh"])
        assert shdr["filter"] == hdr["filter"] and shdr["channels"] == c
        idx = ((r0 + np.arange(nr))[:, None] * cols + (c0 + np.arange(nc))[None, :]).reshape(-1)
        ref = descs[idx]
        assert np.array_equal(sdescs["w"], ref["w"]) and np.array_equal(sdescs["h"], ref["h"])
        assert np.array_equal(sdescs["value"].view(np.uint32), ref["value"].view(np.uint32))
        parts = [pixels[int(d["offset"]):int(d["offset"]) + int(d["w"]) * int(d["h"]) * c] for d in ref]
        assert np.array_equal(spx, np.concatenate(parts))
    # out-of-grid and empty windows
    for win in [(cols, 0, 1, 1), (0, rows, 1, 1), (0, 0, cols + 1, 1), (0, 0, 1, rows + 1), (0, 0, 0, 1), (0, 0, 1, 0),
                (cols - 1, 0, 2, 1)]:
        with pytest.raises(N.PixlzrError) as e:
            N.container_crop(raw, *win)
        assert e.value.status == N.E_ARG, win
    # truncated file, bad line table: PXZ_E_FORMAT from the header check alone
    for bad in [raw[:-1], raw + b"\0", raw[:30]]:
        with pytest.raises(N.PixlzrError) as e:
            N.container_crop(bad, 0, 0, 1, 1)
        assert e.value.status == N.E_FORMAT
        with pytest.raises(N.PixlzrError) as e:
            N.container_header(bad)
        assert e.value.status == N.E_FORMAT
    # row 0 one byte shorter and row 1 one byte longer in the line table (the total still matches): rows 0 and 1 no longer
    # fill their entries, which the crop sees when it walks them
    moved = bytearray(raw)
    l0, l1 = struct.unpack(">II", moved[26:34])
    moved[26:34] = struct.pack(">II", l0 - 1, l1 + 1)
    N.container_header(bytes(moved))  # the sum is intact
    for r0 in (0, 1):
        with pytest.raises(N.PixlzrError) as e:
            N.container_crop(bytes(moved), 0, r0, 1, 1)
        assert e.value.status == N.E_FORMAT
    # a window below the two rows jumps over them by the (wrong but consistent) prefix: row 2 starts where it did
    assert N.container_crop(bytes(moved), 0, 2, cols, 1) == N.container_crop(raw, 0, 2, cols, 1)


def test_corruption_outside_the_window_is_not_read():
    raw = open(os.path.join(GOLDEN, "Big-Ruscher.pix"), "rb").read()
    hdr = N.container_header(raw)
    cols, rows = N.grid(hdr["w"], hdr["h"], hdr["bw"], hdr["bh"])
    line = struct.unpack(f">{rows}I", raw[26:26 + 4 * rows])
    row5 = 26 + 4 * rows + sum(line[:5])  # first record of block row 5
    bad = bytearray(raw)
    bad[row5:row5 + 5] = b"BLOCK"  # a broken record magic
    bad = bytes(bad)
    with pytest.raises(N.PixlzrError):
        N.container_decode(bad)  # the full decoder refuses the file
    good = N.container_crop(bad, 0, 0, cols, 5)  # rows 0..4: never reads row 5
    assert good == N.container_crop(raw, 0, 0, cols, 5)
    assert N.container_crop(bad, 3, 6, 4, rows - 6) == N.container_crop(raw, 3, 6, 4, rows - 6)
    N.container_decode(good)
    for win in [(0, 5, 1, 1), (cols - 1, 5, 1, 1), (0, 4, 2, 2)]:  # the corrupt row is in the window (even a column it skips)
        with pytest.raises(N.PixlzrError) as e:
            N.container_crop(bad, *win)
        assert e.value.status == N.E_FORMAT, win
    # a hostile QOI header inside the window is refused as the full decoder refuses it
    hostile = bytearray(raw)
    qoi = row5 + 13
    hostile[qoi:qoi + 8] = struct.pack(">II", 65535, 65535)
    with pytest.raises(N.PixlzrError):
        N.container_crop(bytes(hostile), 0, 5, 1, 1)
    assert N.container_crop(bytes(hostile), 0, 0, 1, 5) == N.container_crop(raw, 0, 0, 1, 5)


def test_crop_size_query_and_capacity():
    raw = open(os.path.join(GOLDEN, "base.pixlzr"), "rb").read()
    buf = np.frombuffer(raw, np.uint8)
    n = N.lib().pxz_container_crop(N.ptr(buf), buf.size, 2, 3, 4, 5, None, 0)
    want = N.container_crop(raw, 2, 3, 4, 5)
    assert n == len(want)
    out = np.zeros(n, np.uint8)
    assert N.lib().pxz_container_crop(N.ptr(buf), buf.size, 2, 3, 4, 5, N.ptr(out), n - 1) == N.E_ARG
    assert N.lib().pxz_container_crop(N.ptr(buf), buf.size, 2, 3, 4, 5, N.ptr(out), n) == n
    assert out.tobytes() == want


def test_cli_region():
    cli = P.cli
    a = cli.parse_args(["-i", "a.pix", "-o", "b.png", "--region", "10,20,300,40"])
    assert a.region == (10, 20, 300, 40) and cli.region_error(a) is None
    assert cli.parse_args(["-i", "a.pix", "-o", "b.png"]).region is None
    a = cli.parse_args(["-i", "a.pixlzr", "-o", "b.jpg", "--region=0,0,1,1"])
    assert a.region == (0, 0, 1, 1) and cli.region_error(a) is None
    for bad in ["1,2,3", "1,2,3,4,5", "a,b,c,d", "0,0,0,5", "-1,0,4,4"]:
        with pytest.raises(SystemExit):
            cli.parse_args(["-i", "a.pix", "-o", "b.png", "--region", bad])
    for i, o in [("a.png", "b.pix"), ("a.png", "b.png"), ("a.pix", "b.pix"), ("a.pix", "b")]:
        a = cli.parse_args(["-i", i, "-o", o, "--region", "0,0,8,8"])
        assert "--region" in cli.region_error(a)
        with pytest.raises(ValueError, match="--region"):
            cli.run(a)
        assert cli.main(["-i", i, "-o", o, "--region", "0,0,8,8"]) == 2  # refused before any file is opened
