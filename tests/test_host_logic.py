"""CPU-only tests of the product's host side: the C-ABI library loads and exports every symbol the
header declares, the host container stage reproduces the reference's files byte-for-byte, and the
value -> level thresholds agree with the oracle.  No compute calls (no GPU here)."""
import hashlib
import os
import re

import numpy as np
import pytest

import oracle as O
import pixlzr_b200 as P
from conftest import GOLDEN, ROOT, load_png

N = P.native


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "pixlzr_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(pxz_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 30
    lib = N.lib()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} is declared in the header but not exported"
    assert declared == set(N.SYMBOLS), declared ^ set(N.SYMBOLS)
    assert lib.pxz_abi_version() == 1


def test_no_gpu_fails_loudly():
    if N.device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(N.PixlzrError):
        N.Context(0)
    with pytest.raises(N.PixlzrError):
        P.Pixlzr.from_image(np.zeros((8, 8, 3), np.uint8), 4, 4).shrink_by(P.FilterType.Lanczos3, 1.0)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "pixlzr-rust_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cpp", ".cu", ".h", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "pxz_oracle" not in src and "import oracle" not in src and "from oracle" not in src, f


def test_srgb_lut_inc_matches_oracle(golden_meta):
    txt = open(os.path.join(ROOT, "pixlzr-rust_b200", "csrc", "srgb_lut.inc")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    vals = [float.fromhex(t.rstrip("f")) for t in re.findall(r"-?0x[0-9a-f.]+p[+-]?\d+f", txt)]
    arr = np.array(vals, dtype="<f4")
    assert arr.shape == (256,)
    assert hashlib.sha256(arr.tobytes()).hexdigest() == golden_meta["kat"]["srgb_lut_sha256_le_f32"]
    assert np.array_equal(arr, O.srgb_lut())


def test_grid_and_filter_enum():
    assert N.grid(1080, 1617, 64, 64) == (17, 26)
    assert N.grid(1920, 1080, 32, 32) == (60, 34)
    assert N.grid(7680, 4320, 64, 64) == (120, 68)
    assert N.grid(5, 5, 64, 64) == (1, 1)
    assert [int(f) for f in P.FilterType] == [0, 1, 2, 3, 4]
    assert P.FilterType.from_u8(200) == P.FilterType.Nearest and P.FilterType.from_u8(4) == P.FilterType.Lanczos3


def test_parse_shrinking_factor(golden_meta):
    """src/bin/main.rs:281-297"""
    for s, want in golden_meta["kat"]["parse_shrinking_factor"].items():
        assert P.parse_shrinking_factor(s) == want, s


def test_level_thresholds_match_oracle(golden_meta):
    for v, exp in golden_meta["kat"]["level_dims_64_56_17"].items():
        got = [N.reduce_dims(float(v), float(v), n, n)[0] for n in (64, 56, 17)]
        assert got == exp, v
    # +-4096 ulps around every boundary 2^(k - 1/2), k = 0..-20, against log2f/round themselves
    for k in range(0, 21):
        centre = np.float32(2.0 ** (-k - 0.5))
        bits = int(centre.view(np.uint32))
        cand = np.arange(bits - 4096, bits + 4096, dtype=np.uint32).view(np.float32)
        for v in cand[::37].tolist() + cand[4096 - 40:4096 + 40].tolist():
            a = N.reduce_dims(v, v, 65535, 40000)
            b = O.reduce_dims(v, v, 65535, 40000)
            assert a[:2] == b[:2], (k, v)
            assert np.float32(a[2]) == np.float32(b[2])
    # specials
    for v in [0.0, -0.0, -0.25, -1.0, -1.5, float("inf"), float("nan"), 1e-30, 3.0, -5.0]:
        a, b = N.reduce_dims(v, 0.3, 64, 17), O.reduce_dims(v, 0.3, 64, 17)
        assert a[:2] == b[:2], v
        assert (np.isnan(a[2]) and np.isnan(b[2])) or a[2] == b[2], v


def test_container_decode_encode_golden_files():
    for name in ("Big-Ruscher.pix", "base.pixlzr"):
        raw = open(os.path.join(GOLDEN, name), "rb").read()
        hdr, descs, pixels = N.container_decode(raw)
        ref, filt = O.container_decode(raw)
        assert (hdr["w"], hdr["h"], hdr["bw"], hdr["bh"], hdr["channels"], hdr["filter"]) == \
               (ref.width, ref.height, ref.block_width, ref.block_height, ref.channels, filt)
        assert np.array_equal(descs, ref.descs.astype(N.DESC_DTYPE))
        assert np.array_equal(pixels, ref.payload)
        again = N.container_encode(hdr["w"], hdr["h"], hdr["bw"], hdr["bh"], hdr["filter"], hdr["channels"], descs,
                                   pixels, None, nthreads=4)
        assert again == raw, name


def test_from_image_encode_equals_base_pixlzr():
    """benches/base.png --from_image(64,64)+save--> benches/base.pixlzr, byte for byte (host only)."""
    img = load_png("base.png")
    pix = P.Pixlzr.from_image(img, 64, 64)
    assert pix.block_grid_dimensions() == (17, 26)
    assert pix.block_grid_has_trailing() == (True, True)
    blocks = pix.blocks
    assert len(blocks) == 442 and all(b.block_value is None for b in blocks)
    assert blocks[16].dimensions() == (56, 64) and blocks[-1].dimensions() == (56, 17)
    assert pix.encode_to_vec() == open(os.path.join(GOLDEN, "base.pixlzr"), "rb").read()


def test_decode_from_vec_mirrors_reference():
    pix = P.Pixlzr.decode_from_vec(open(os.path.join(GOLDEN, "Big-Ruscher.pix"), "rb").read())
    assert pix.dimensions() == (1920, 1080) and pix.block_dimensions() == (32, 32)
    assert pix.filter == P.FilterType.Nearest and not pix.has_alpha()
    blocks = pix.blocks
    assert len(blocks) == 2040 and all(b.block_value is not None for b in blocks)
    assert np.float32(blocks[0].block_value) == np.float32(float.fromhex("0x1.76b0acp-9"))
    # already-valued blocks are skipped by shrink_by (pixlzr.rs:168-170): no GPU needed, no change
    before = pix.encode_to_vec()
    pix.shrink_by(P.FilterType.Lanczos3, 1.0)
    assert pix.encode_to_vec() == before


def test_container_rejects_garbage():
    with pytest.raises(N.PixlzrError):
        N.container_decode(b"NOTPIX" + bytes(40))
    raw = open(os.path.join(GOLDEN, "Big-Ruscher.pix"), "rb").read()
    with pytest.raises(N.PixlzrError):
        N.container_decode(raw[:-5])
    with pytest.raises(N.PixlzrError):
        N.container_decode(raw + b"\0")


def _tiny_container(w, h, bw, bh, blocks):
    """A v0.0.2 container from (qoi_w, qoi_h, qoi_body_ops) per block, all in one block row per grid row."""
    import struct
    cols = -(-w // bw)
    rows = -(-h // bh)
    enc = []
    for (qw, qh, ops) in blocks:
        body = struct.pack(">IIBB", qw, qh, 4, 0) + ops + bytes(7) + b"\x01"
        enc.append(b"block" + struct.pack(">f", 0.5) + struct.pack(">I", len(body)) + body)
    lines = [b"".join(enc[r * cols:(r + 1) * cols]) for r in range(rows)]
    head = b"PIXLZR" + bytes([0, 0, 2, 0]) + struct.pack(">IIII", w, h, bw, bh)
    return head + b"".join(struct.pack(">I", len(ln)) for ln in lines) + b"".join(lines)


def test_container_hostile_files_are_refused():
    """ADVICE r1: truncated QOI streams, blocks that claim more pixels than their stream can hold, grids that differ
    between the reference's f32 arithmetic and integers, block rows that do not fill their line-table entry."""
    rgba = b"\xff\x10\x20\x30\xff"                      # QOI_OP_RGBA: one pixel
    ok = _tiny_container(2, 1, 1, 1, [(1, 1, rgba), (1, 1, rgba)])
    hdr, descs, pixels = N.container_decode(ok)
    assert (hdr["w"], hdr["h"]) == (2, 1) and pixels.tolist() == [0x10, 0x20, 0x30, 0xFF] * 2
    # a 2x2 block whose stream holds one pixel: the qoi crate stops with UnexpectedBufferEnd, so do we
    with pytest.raises(N.PixlzrError):
        N.container_decode(_tiny_container(2, 2, 2, 2, [(2, 2, rgba)]))
    # 31 bytes that claim 65535 x 65535 pixels: refused before anything of that size is allocated
    with pytest.raises(N.PixlzrError):
        N.container_decode(_tiny_container(1, 1, 1, 1, [(65535, 65535, rgba)]))
    # a run can fill a block: 1 op byte -> up to 62 pixels
    run = _tiny_container(8, 4, 8, 4, [(8, 4, rgba + b"\xde")])     # RGBA + RUN(31) = 32 pixels
    assert N.container_decode(run)[2].size == 8 * 4 * 4
    # w = 2^24 + 1: ceil in f32 gives 512 columns of 32768, integers give 513 -> refused
    with pytest.raises(N.PixlzrError):
        N.container_decode(_tiny_container(16777217, 1, 32768, 1, [(1, 1, rgba)] * 512))
    # line table says 1 byte less for row 0 and 1 more for row 1 (the sum still matches the file)
    two = bytearray(_tiny_container(1, 2, 1, 1, [(1, 1, rgba), (1, 1, rgba)]))
    import struct
    l0, l1 = struct.unpack(">II", two[26:34])
    two[26:34] = struct.pack(">II", l0 - 1, l1 + 1)
    with pytest.raises(N.PixlzrError):
        N.container_decode(bytes(two))


def test_pixlzrblock_accessors():
    """block.rs:346-399"""
    b = P.PixlzrBlock(np.zeros((100, 100, 4), np.uint8))
    assert b.width == 100 and b.height == 100 and b.has_alpha()
    px = b.pixels()
    assert px.shape == (10000, 4)
    same = b.resize(100, 100, P.FilterType.Lanczos3)  # same size: clone, no GPU involved
    assert same.data is not b.data and np.array_equal(same.data, b.data)


@pytest.mark.parametrize("filt", range(5))
def test_resample_tables_match_oracle_bit_for_bit(filt):
    """The host-built tap tables the kernels apply are the image-crate weights of the oracle, bit for bit."""
    pairs = [(64, 64), (64, 32), (64, 16), (64, 8), (64, 4), (64, 2), (64, 1), (56, 28), (56, 7), (17, 9), (17, 3), (32, 64),
             (16, 64), (8, 64), (1, 64), (2, 56), (28, 56), (9, 17), (3, 2), (5, 200), (200, 3), (1, 1), (100, 10)]
    for n_in, n_out in pairs:
        l0, c0, w0 = O.axis_weights(n_in, n_out, filt)
        l1, c1, w1 = N.resample_table(n_in, n_out, filt)
        assert np.array_equal(l0, l1) and np.array_equal(c0, c1), (n_in, n_out)
        assert w0.shape == w1.shape and np.array_equal(w0.view(np.uint32), w1.view(np.uint32)), (n_in, n_out)


def test_cli_arguments_and_operation_selection():
    """src/bin/main.rs:7-114: flags, defaults, extension-based operation selection."""
    import pixlzr_b200 as P
    cli = P.cli
    a = cli.parse_args(["-i", "a.png", "-o", "b.pix"])
    assert (a.block_width, a.block_height, a.shrinking_factor, a.filter, a.direction_wise, a.force) == (64, None, "1", "lanczos3", None, False)
    a = cli.parse_args(["-i", "a.png", "-o", "b.png", "-b", "32", "--block-height", "16", "-k", "-1/2", "-f", "catmull-rom",
                                       "-d", "true", "--force"])
    assert (a.block_width, a.block_height, a.shrinking_factor, a.filter, a.direction_wise, a.force) == (32, 16, "-1/2", "catmull-rom", True, True)
    assert P.parse_shrinking_factor(a.shrinking_factor) == -0.5
    assert cli.operation("x.png", "y.pix") == ("image", "pix")
    assert cli.operation("x.PIXLZR", "y.jpg") == ("pix", "image")
    assert cli.operation("x.pix", "y.PiX") == ("pix", "pix")
    assert cli.operation("x", "y") == ("image", "pix")          # no extension: image in, container out (main.rs:100, 109)
    assert cli.operation("x.webp", "y.png") == ("image", "image")
    assert set(cli.FILTERS) == {"nearest", "triangle", "catmull-rom", "gaussian", "lanczos3"}


# ---------------------------------------------------------------------------------------------
# per-block filter pairs (SURVEY.md §8f N4): the table of the reference's experiment log
# ---------------------------------------------------------------------------------------------
def test_strategy_table_matches_reference_log():
    """pxz_strategy_by_level (host function, no GPU) and the oracle's table against tests/golden/strategies.json, which
    tests/golden/make_strategy_fixture.py parsed from strategies.txt / strategies_by_level.txt."""
    import json
    with open(os.path.join(GOLDEN, "strategies.json")) as f:
        fx = json.load(f)
    down, up = P.native.strategy_by_level()
    odown, oup = O.strategy_by_level()
    assert down.size == up.size == P.native.STRATEGY_BUCKETS == O.STRATEGY_BUCKETS == 65
    assert np.array_equal(down, odown) and np.array_equal(up, oup)
    for b, (d, u) in fx["per_bucket"].items():  # every bucket the author measured
        b = min(int(b), 64)  # the log goes beyond v = 1; all of those are (Nearest, Nearest) like bucket 64
        assert (down[b], up[b]) == (d, u), b
    for r in fx["ranges"]:  # the summary: ranges of v
        lo = int(round(r["lo"] * 64))
        hi = 65 if r["hi"] is None else int(round(r["hi"] * 64))
        assert (down[lo:hi] == r["down"]).all() and (up[lo:hi] == r["up"]).all(), r


def test_strategy_bucket_rule():
    """bucket = floor(64 * value / sqrt(2)) in f32, clamped; the library and the oracle agree on every edge."""
    f32 = np.float32
    vals = [0.0, -0.0, -1.0, float("nan"), float("inf"), 1e-30, 0.0221, 0.5, 0.99436, 1.0, 1.4142135, 1.4142137, 5.0]
    vals += list(np.nextafter(f32(k / 64 * 2 ** 0.5), f32(s)) for k in range(1, 65) for s in (0, 4))
    rng = np.random.default_rng(3)
    vals += list(rng.random(2000, dtype=np.float32) * 1.6)
    for v in vals:
        b = P.native.strategy_bucket(v)
        assert b == O.strategy_bucket(v)
        t = f32(v) * f32(45.25483322143555)
        want = 0 if not (t > 0) else (64 if t >= 64 else int(t))
        assert b == want, (v, b, want)
    with pytest.raises(ValueError):
        P.native.Context.set_strategy(None, np.zeros(3, np.uint8), np.zeros(65, np.uint8))


def test_merge_shard_containers_host():
    """Block-row shard files stitch to the image's file (host stage only; the device path is tested under -m gpu)."""
    S = P.sharding
    rng = np.random.default_rng(4)
    w, h, bs = 150, 210, 32  # 7 block rows, the last one partial
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    img[40:120, 10:90] = (9, 200, 77)
    whole = O.container_encode(O.shrink(img, bs, bs, O.METRIC_OKLAB_MAD, 0.02, O.LANCZOS3), 4)
    for world in (1, 2, 3, 7, 9):  # 9 ranks: two of them hold no block row
        files = []
        for rank in range(world):
            y0, y1 = S.shard_pixel_rows(h, bs, world, rank)
            files.append(O.container_encode(O.shrink(np.ascontiguousarray(img[y0:y1]), bs, bs, O.METRIC_OKLAB_MAD, 0.02, O.LANCZOS3), 4)
                         if y1 > y0 else b"")
        assert S.merge_shard_containers(files, w, h) == whole, world
    with pytest.raises(ValueError):
        S.merge_shard_containers([files[0]], w, h)          # rows missing
    with pytest.raises(ValueError):
        S.merge_shard_containers([b"garbage" * 5], w, h)
    with pytest.raises(ValueError):
        S.merge_shard_containers([b"", b""], w, h)
    with pytest.raises(ValueError):
        S.merge_shard_containers(files[::-1], w, h)         # the partial row must come last


def test_interleaved_block_row_shards_host():
    """Interleaved layout (block row g -> rank g mod world): merged descriptors / payload / container file equal the
    single-process result, for worlds with and without empty ranks and a partial last block row."""
    S = P.sharding
    assert S.cyclic_block_rows(10, 4, 1) == [1, 5, 9] and S.cyclic_block_rows(3, 8, 5) == []
    assert sorted(sum((S.cyclic_block_rows(1024, 8, r) for r in range(8)), [])) == list(range(1024))
    rng = np.random.default_rng(4)
    w, h, bs = 150, 210, 32  # 7 block rows, the last one partial
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    img[40:120, 10:90] = (9, 200, 77)
    whole = O.shrink(img, bs, bs, O.METRIC_OKLAB_MAD, 0.02, O.LANCZOS3)
    whole_file = O.container_encode(whole, 4)
    cols, rows = O.grid(w, h, bs, bs)[0], -(-h // bs)
    for world in (1, 2, 3, 7, 9):
        parts, files = [], []
        back = np.zeros_like(img)
        for rank in range(world):
            idx = S.cyclic_block_rows(rows, world, rank)
            local = S.gather_block_rows(img, bs, idx)
            S.scatter_block_rows(local, back, bs, idx)
            if local.shape[0]:
                sh = O.shrink(local, bs, bs, O.METRIC_OKLAB_MAD, 0.02, O.LANCZOS3)
                parts.append((sh.descs, sh.payload))
                files.append(O.container_encode(sh, 4))
            else:
                parts.append((np.zeros(0, P.native.DESC_DTYPE), np.zeros(0, np.uint8)))
                files.append(b"")
        assert np.array_equal(back, img)
        descs, pixels = S.merge_shards_cyclic(parts, cols)
        assert np.array_equal(descs, whole.descs.astype(descs.dtype)) and np.array_equal(pixels, whole.payload), world
        assert S.merge_shard_containers_cyclic(files, w, h) == whole_file, world
    with pytest.raises(ValueError):
        S.merge_shard_containers_cyclic([files[0]], w, h)
    with pytest.raises(ValueError):
        S.merge_shard_containers_cyclic([b"garbage" * 5], w, h)
    # 7 rows over 3 ranks = 3 + 2 + 2: with ranks 0 and 2 swapped the first rank runs out of rows
    p3 = []
    for rank in range(3):
        sh = O.shrink(S.gather_block_rows(img, bs, S.cyclic_block_rows(rows, 3, rank)), bs, bs, O.METRIC_OKLAB_MAD, 0.02, O.LANCZOS3)
        p3.append((sh.descs, sh.payload))
    with pytest.raises(ValueError):
        S.merge_shards_cyclic([p3[2], p3[1], p3[0]], cols)


def test_bench_device_frames_do_not_depend_on_the_shard_layout():
    """bench.py generates the gigapixel frame of C4 per rank: rows [y0, y1) in the contiguous layout, the rank's own block
    rows in the interleaved one.  Both must be cuts of ONE frame (the checksum comparison across layouts and rank counts
    relies on it) — checked here on the CPU device with a small frame whose last block row is partial."""
    import sys

    import torch

    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench

    S = P.sharding
    w, h = 192, 64 * 5 + 24
    whole = bench.synth_rows_device(torch, 0, h, w, 7, "cpu").numpy()
    assert whole.shape == (h, w, 4) and (whole[..., 3] == 255).all()
    a = bench.synth_rows_device(torch, 128, 256, w, 7, "cpu").numpy()
    assert np.array_equal(a, whole[128:256])
    rows = -(-h // 64)
    for world in (2, 3):
        back = np.zeros_like(whole)
        for rank in range(world):
            idx = S.cyclic_block_rows(rows, world, rank)
            local = bench.synth_block_rows_device(torch, idx, h, w, 7, "cpu").numpy()
            assert np.array_equal(local, S.gather_block_rows(whole, 64, idx))
            S.scatter_block_rows(local, back, 64, idx)
        assert np.array_equal(back, whole)


def test_bench_dump_outputs_is_a_fixed_sample_within_the_budget(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 / float64 files within the byte budget, every descriptor, and pixels sampled at the
    same positions in every frame and in every run, so that two builds can be compared file for file."""
    import sys

    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench

    h, w, n = 96, 160, 3
    pos = np.arange(h * w)
    # pixel p of frame f is (p mod 256, p div 256, f, 255): a sampled pixel tells where it came from
    frames = [np.stack([pos % 256, pos // 256, np.full(h * w, f), np.full(h * w, 255)], -1).astype(np.uint8).reshape(h, w, 4)
              for f in range(n)]
    rng = np.random.default_rng(6)
    descs = []
    for _ in range(n):
        d = np.zeros(15, N.DESC_DTYPE)
        d["offset"], d["value"] = np.cumsum(rng.integers(1, 1 << 20, 15)), rng.random(15, dtype=np.float32)
        d["w"], d["h"] = rng.integers(1, 65, 15), rng.integers(1, 65, 15)
        descs.append(d)
    payloads = [rng.integers(0, 256, size, dtype=np.uint8) for size in (5000, 7000, 6000)]
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 16)
    total = bench.dump_outputs(str(tmp_path / "a"), frames, descs, payloads)
    bench.dump_outputs(str(tmp_path / "b"), frames, descs, payloads)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b")) and len(names) == 7
    out = {}
    for name in names:
        a, b = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), name
        out[name[:-4]] = a
    assert sum(a.nbytes for a in out.values()) == total <= 1 << 16
    for field, name in (("offset", "block_offset"), ("value", "block_value"), ("w", "block_width"), ("h", "block_height")):
        assert np.array_equal(out[name], np.stack([d[field] for d in descs]).astype(out[name].dtype)), name
    assert out["payload_bytes"].tolist() == [5000, 7000, 6000]
    assert out["payload_sample"].shape[0] == n and 0 < out["payload_sample"].shape[1] <= 5000
    dec = out["decoded_sample"]
    assert dec.shape[0] == n and 0 < dec.shape[1] < h * w and dec.shape[2] == 4
    where = dec[..., 0] + 256 * dec[..., 1]
    assert (np.diff(where[0]) > 0).all() and (where == where[0]).all()
    assert (dec[..., 2] == np.arange(n)[:, None]).all() and (dec[..., 3] == 255).all()
