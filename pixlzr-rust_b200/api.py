"""Host-side mirror of the reference's public API for the hot path, on top of the C ABI.

Same names, argument meaning and error behaviour as crate `pixlzr` v0.3.1 (citations are relative
to the reference tree), so the parity tests read like the reference's own:

    Pixlzr::from_image / shrink_by / shrink_directionally / expand / to_image
        src/data_types/pixlzr.rs:77-205, pixlzr_image.rs:6-74
    Pixlzr::encode_to_vec / decode_from_vec / open / save     src/encoding/mod.rs:40-165, src/io.rs:79-96
    PixlzrBlock::resize                                        src/data_types/block.rs:273-334
    get_block_variance(_directionally), reduce_image_section   src/operations.rs:26-259
    process / process_custom                                   src/process/mod.rs:31-121
    FilterType                                                 src/data_types/mod.rs:10-30,110-121
    parse_shrinking_factor                                     src/bin/main.rs:47-68

Images are numpy uint8 arrays of shape (H, W, 3|4) (what `image::DynamicImage` holds for RGB8 /
RGBA8).  All pixel work runs on the GPU through libpixlzr_b200.so; where the reference panics this
raises.  Resampling follows the reference's `image`-crate branch (block.rs:282-290), the only one
its fixtures pin (DESIGN.md).
"""
from __future__ import annotations

import enum
import os
from contextlib import contextmanager
from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from . import _native as N

BASE_FACTOR = 10.0  # pixlzr.rs:15


class FilterType(enum.IntEnum):
    """#[repr(u8)] enum, src/data_types/mod.rs:10-30."""

    Nearest = 0
    Triangle = 1
    CatmullRom = 2
    Gaussian = 3
    Lanczos3 = 4

    @classmethod
    def from_u8(cls, value: int) -> "FilterType":
        """impl From<u8> (mod.rs:110-121): unknown values map to Nearest."""
        return cls(value) if 0 <= value <= 4 else cls.Nearest


_default_ctx: Optional[N.Context] = None


def default_context() -> N.Context:
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = N.Context(int(os.environ.get("PXZ_DEVICE", "0")))
    return _default_ctx


@dataclass
class PixlzrBlock:
    """PixlzrBlockRaw (block.rs:76-81): tightly packed pixels + optional block value."""

    data: np.ndarray  # (h, w, 3|4) uint8
    block_value: Optional[float] = None

    @property
    def width(self) -> int:
        return self.data.shape[1]

    @property
    def height(self) -> int:
        return self.data.shape[0]

    def dimensions(self) -> Tuple[int, int]:
        return self.width, self.height

    def has_alpha(self) -> bool:
        return self.data.shape[2] == 4

    def as_slice(self) -> bytes:
        return np.ascontiguousarray(self.data).tobytes()

    def pixels(self) -> np.ndarray:
        """chunks_exact(3 + alpha) over the raw bytes (block.rs:260-271)."""
        return np.ascontiguousarray(self.data).reshape(-1, self.data.shape[2])

    def resize(self, width: int, height: int, filter: FilterType, ctx: Optional[N.Context] = None) -> "PixlzrBlock":
        """PixlzrBlock::resize (block.rs:273-290): same size -> clone, else resample; value reset to None."""
        if (width, height) == self.dimensions():
            return PixlzrBlock(self.data.copy(), self.block_value)
        if width <= 0 or height <= 0:
            raise ValueError("resize target must be at least 1x1")
        ctx = ctx or default_context()
        c = self.data.shape[2]
        descs = np.zeros(1, N.DESC_DTYPE)
        descs[0] = (0, 0.0, self.width, self.height)
        pl = ctx.payload_upload(width, height, width, height, c, descs, np.ascontiguousarray(self.data).reshape(-1))
        try:
            return PixlzrBlock(pl.expand(int(filter)), None)
        finally:
            pl.free()


def _check_image(image: np.ndarray) -> np.ndarray:
    if not (isinstance(image, np.ndarray) and image.dtype == np.uint8 and image.ndim == 3 and image.shape[2] in (3, 4)):
        raise TypeError("image must be a uint8 array of shape (H, W, 3) or (H, W, 4)")
    if image.shape[0] == 0 or image.shape[1] == 0:
        raise ValueError("empty image")
    return np.ascontiguousarray(image)


@contextmanager
def _on_device(image, ctx: N.Context):
    """`image` as a device image: a device image as it is, a numpy image uploaded for the block and freed after it."""
    if isinstance(image, N.Image):
        yield image
        return
    img = ctx.image_upload(_check_image(image))
    try:
        yield img
    finally:
        img.free()


def _check_rect(width: int, height: int, x: int, y: int, w: int, h: int) -> None:
    """The rectangle errors of pxz_expand_region, raised before anything is read or uploaded."""
    if w <= 0 or h <= 0:
        raise N.PixlzrError(N.E_ARG, "empty rectangle")
    if x < 0 or y < 0 or x + w > width or y + h > height:
        raise N.PixlzrError(N.E_ARG, "rectangle outside the image")


def _touched_blocks(bw: int, bh: int, x: int, y: int, w: int, h: int) -> Tuple[int, int, int, int]:
    """(c0, r0, nc, nr): the block window a pixel rectangle touches."""
    c0, r0 = x // bw, y // bh
    return c0, r0, (x + w - 1) // bw - c0 + 1, (y + h - 1) // bh - r0 + 1


@dataclass
class Strategy:
    """(down, up) filter per value bucket of width 1/64 (pxz_strategy, include/pixlzr_b200.h).  The bucket of a block
    is `Strategy.bucket(block_value)` = floor(64 * value / sqrt(2)) clamped to [0, 64]."""
    down: np.ndarray
    up: np.ndarray

    @classmethod
    def by_level(cls) -> "Strategy":
        """The table the reference's log arrives at (strategies_by_level.txt:1-12)."""
        return cls(*N.strategy_by_level())

    @classmethod
    def uniform(cls, down: FilterType, up: FilterType) -> "Strategy":
        return cls(np.full(N.STRATEGY_BUCKETS, int(down), np.uint8), np.full(N.STRATEGY_BUCKETS, int(up), np.uint8))

    @staticmethod
    def bucket(value: float) -> int:
        return N.strategy_bucket(value)

    @classmethod
    def fit(cls, images, block_width: int, block_height: int, factor: float, directionally: bool = False,
            exact_values: bool = False, base: Optional["Strategy"] = None,
            ctx: Optional[N.Context] = None) -> Tuple["Strategy", "StrategyReport"]:
        """EXTENSION: the table of least summed error over `images` (numpy images) for shrink_by (or shrink_directionally)
        with `factor` at this block size: every (down, up) pair is measured on the device per value bucket
        (pxz_strategy_measure), the reports are added and each bucket takes its best pair (pxz_strategy_choose; ties and
        empty buckets keep `base`'s pair, default by_level).  Returns the table and the summed report; report.total(table)
        is the exact error of the table's decodes in the default resample arithmetic."""
        ctx = ctx or default_context()
        metric = N.METRIC_SOBEL_DIR if directionally else N.METRIC_OKLAB_MAD
        flags = N.FLAG_EXACT_VALUES if exact_values else 0
        sse = np.zeros((N.STRATEGY_BUCKETS, N.FILTER_PAIRS), np.uint64)
        blocks = np.zeros(N.STRATEGY_BUCKETS, np.uint32)
        for image in images:
            img = ctx.image_upload(_check_image(image))
            try:
                s, b = img.strategy_measure(block_width, block_height, metric, factor, flags)
            finally:
                img.free()
            sse += s
            blocks += b
        down, up = N.strategy_choose(sse, blocks, None if base is None else (base.down, base.up))
        return cls(down, up), StrategyReport(sse, blocks)


@dataclass
class StrategyReport:
    """What pxz_strategy_measure returns (summed over images): sse[bucket, down * 5 + up] = the squared error of the blocks
    of that bucket when shrunk with `down` and expanded with `up`; blocks[bucket] = how many blocks the bucket holds."""
    sse: np.ndarray     # uint64 [65, 25]
    blocks: np.ndarray  # uint32 [65]

    def total(self, strategy: Strategy) -> int:
        """The squared error of a decode with `strategy` installed: the sum of each bucket's entry for its pair."""
        pairs = strategy.down.astype(np.int64) * 5 + strategy.up.astype(np.int64)
        return int(sum(int(self.sse[b, pairs[b]]) for b in range(N.STRATEGY_BUCKETS)))


def psnr_of(total_sse: int, samples: int) -> float:
    """10 log10(255^2 * samples / total_sse) in dB (samples = width * height * channels); inf for identical images."""
    if total_sse == 0:
        return float("inf")
    return 10.0 * float(np.log10(255.0 * 255.0 * samples / float(total_sse)))


def sse_budget(psnr: float, samples: int) -> int:
    """The largest squared error whose psnr_of(..., samples) is >= `psnr` dB: the formula's value, then corrected by single
    steps against psnr_of itself, so that the two never disagree (0 for a target of inf: only an exact decode reaches it)."""
    psnr = float(psnr)
    if psnr != psnr or samples <= 0:
        raise ValueError("a PSNR target needs a number of dB and a positive sample count")
    top = 2 ** 64 - 1  # the budget is a u64
    with np.errstate(over="ignore", divide="ignore"):
        bound = np.float64(255.0 * 255.0 * samples) / np.power(np.float64(10.0), psnr / 10.0)
    budget = top if not bound < top else int(np.floor(bound))
    while budget < top and psnr_of(budget + 1, samples) >= psnr:
        budget += 1
    while budget > 0 and psnr_of(budget, samples) < psnr:
        budget -= 1
    return budget


@dataclass
class RateDistortion:
    """EXTENSION (pxz_rd_curve): every distinct payload a factor gives, in increasing factor.  factor[i] is the smallest f32
    factor giving payload i, bytes[i] its payload bytes (strictly increasing), sse[i] the squared error of its decode against
    the source; a factor between factor[i] and factor[i + 1] gives payload i."""
    factor: np.ndarray  # float32 [n]
    bytes: np.ndarray   # uint64 [n]
    sse: np.ndarray     # uint64 [n]
    samples: int        # width * height * channels of the source

    @property
    def psnr(self) -> np.ndarray:
        return np.array([psnr_of(int(e), self.samples) for e in self.sse], np.float64)

    def smallest_within(self, max_sse: int) -> Optional[int]:
        """Index of the smallest payload whose error is at most `max_sse` (the point pxz_shrink_to_error picks), None if no
        factor reaches it."""
        ok = np.nonzero(self.sse <= np.uint64(max_sse))[0]
        return int(ok[0]) if ok.size else None


def rd_curve(image, block_width: int, block_height: int, filter_down: FilterType, filter_up: FilterType, directionally: bool = False,
             ctx: Optional[N.Context] = None) -> RateDistortion:
    """EXTENSION: the exact (bytes, squared error) curve of shrink_by (or shrink_directionally) with `filter_down` and a decode
    with `filter_up`, over every finite factor, computed on the device (numpy or device image)."""
    ctx = ctx or (image.ctx if isinstance(image, N.Image) else default_context())
    with _on_device(image, ctx) as img:
        metric = N.METRIC_SOBEL_DIR if directionally else N.METRIC_OKLAB_MAD
        factor, nbytes, sse = img.rd_curve(block_width, block_height, metric, int(filter_down), int(filter_up), 0)
        return RateDistortion(factor, nbytes, sse, img.w * img.h * img.c)


@dataclass
class OptimalCurve:
    """EXTENSION (pxz_rdo_curve): the rate-distortion optimised curve, every block free to take the dims of any level pair.
    Point 0 has every block at 1 x 1; bytes strictly increases, sse strictly decreases and the last point has sse 0.  No choice of
    block sizes has at most bytes[i] payload bytes and less error than sse[i]."""
    bytes: np.ndarray   # uint64 [n]
    sse: np.ndarray     # uint64 [n]
    samples: int        # width * height * channels of the source

    @property
    def psnr(self) -> np.ndarray:
        return np.array([psnr_of(int(e), self.samples) for e in self.sse], np.float64)

    def best_within(self, max_bytes: int) -> Optional[int]:
        """Index of the least error within `max_bytes` payload bytes (the point pxz_rdo_shrink_to_size picks), None if even
        point 0 is larger."""
        ok = np.nonzero(self.bytes <= np.uint64(max_bytes))[0]
        return int(ok[-1]) if ok.size else None

    def smallest_within(self, max_sse: int) -> Optional[int]:
        """Index of the fewest bytes whose error is at most `max_sse` (the point pxz_rdo_shrink_to_error picks)."""
        ok = np.nonzero(self.sse <= np.uint64(max_sse))[0]
        return int(ok[0]) if ok.size else None


def rdo_curve(image, block_width: int, block_height: int, filter_down: FilterType, filter_up: FilterType,
              ctx: Optional[N.Context] = None) -> OptimalCurve:
    """EXTENSION: the rate-distortion optimised (bytes, squared error) curve of an image when each block's size is chosen on its
    own, shrunk with `filter_down` and decoded with `filter_up`, computed on the device (numpy or device image)."""
    ctx = ctx or (image.ctx if isinstance(image, N.Image) else default_context())
    with _on_device(image, ctx) as img:
        nbytes, sse = img.rdo_curve(block_width, block_height, int(filter_down), int(filter_up))
        return OptimalCurve(nbytes, sse, img.w * img.h * img.c)


@dataclass
class ErrorReport:
    """EXTENSION: the error of one image against another, per block of a grid (pxz_image_error)."""
    block_sse: np.ndarray  # uint64 [rows, cols]: sum of (a - b)^2 over the tile's pixels and channels
    block_max: np.ndarray  # uint8 [rows, cols]: max |a - b| over the same
    total_sse: int
    samples: int           # width * height * channels

    @property
    def mse(self) -> float:
        return self.total_sse / self.samples

    @property
    def psnr(self) -> float:
        return psnr_of(self.total_sse, self.samples)

    @property
    def max_error(self) -> int:
        return int(self.block_max.max()) if self.block_max.size else 0


def image_error(a, b, block_width: int, block_height: int, ctx: Optional[N.Context] = None) -> ErrorReport:
    """EXTENSION: per-block squared error and largest difference of `a` against `b` (numpy images or device images of one
    geometry), computed on the device in one streaming pass; only the per-block figures come back."""
    ctx = ctx or (a.ctx if isinstance(a, N.Image) else default_context())
    with _on_device(a, ctx) as da, _on_device(b, ctx) as db:
        sse, mx, total = da.error(db, block_width, block_height)
        return ErrorReport(sse, mx, total, da.w * da.h * da.c)


def payload_error(payload: N.Payload, source, filter_up: FilterType) -> ErrorReport:
    """EXTENSION: the error of a payload's decode with `filter_up` against its source image (numpy or device image), on the
    payload's block grid (Payload.error): the decode stays on the device."""
    with _on_device(source, payload.ctx) as src:
        sse, mx, total = payload.error(src, int(filter_up))
        return ErrorReport(sse, mx, total, src.w * src.h * src.c)


class Pixlzr:
    """struct Pixlzr (pixlzr.rs:17-25).  Holds either the source image (blocks = tiles, no values) or
    a packed block payload (descriptor table + pixels), both on the host; the GPU does the work."""

    def __init__(self, width, height, block_width, block_height, filter: Optional[FilterType] = None):
        self.width, self.height = width, height
        self.block_width, self.block_height = block_width, block_height
        self.filter = filter
        self._image: Optional[np.ndarray] = None     # set by from_image until the first shrink
        self._descs: Optional[np.ndarray] = None     # N.DESC_DTYPE, row-major
        self._pixels: Optional[np.ndarray] = None    # packed payload
        self._values_present = False
        self._channels = 3
        self.ctx: Optional[N.Context] = None

    # ---- geometry (pixlzr.rs:28-56) ---------------------------------------------------------------
    def dimensions(self):
        return self.width, self.height

    def block_dimensions(self):
        return self.block_width, self.block_height

    def block_grid_width(self) -> int:
        return int(np.ceil(np.float32(self.width) / np.float32(self.block_width)))

    def block_grid_height(self) -> int:
        return int(np.ceil(np.float32(self.height) / np.float32(self.block_height)))

    def block_grid_dimensions(self):
        return self.block_grid_width(), self.block_grid_height()

    def block_grid_has_trailing(self):
        return self.width % self.block_width > 0, self.height % self.block_height > 0

    def has_alpha(self) -> bool:
        return self._channels == 4

    def _ctx(self) -> N.Context:
        if self.ctx is None:
            self.ctx = default_context()
        return self.ctx

    # ---- construction -----------------------------------------------------------------------------
    @classmethod
    def from_image(cls, image: np.ndarray, block_width: int, block_height: int, ctx: Optional[N.Context] = None) -> "Pixlzr":
        """Pixlzr::from_image (pixlzr_image.rs:6-22).  No per-block copies: a block is a window."""
        image = _check_image(image)
        if block_width <= 0 or block_height <= 0:
            raise ValueError("block size must be positive")
        p = cls(image.shape[1], image.shape[0], block_width, block_height, None)
        p._image = image
        p._channels = image.shape[2]
        p.ctx = ctx
        return p

    def _materialise_tiles(self):
        """Turns the window view into an explicit full-size payload (what the reference always holds)."""
        if self._descs is not None:
            return
        img = self._image
        cols, rows = N.grid(self.width, self.height, self.block_width, self.block_height)
        descs = np.zeros(cols * rows, N.DESC_DTYPE)
        parts, off = [], 0
        for by in range(rows):
            for bx in range(cols):
                blk = img[by * self.block_height:(by + 1) * self.block_height,
                          bx * self.block_width:(bx + 1) * self.block_width]
                descs[by * cols + bx] = (off, 0.0, blk.shape[1], blk.shape[0])
                parts.append(np.ascontiguousarray(blk).reshape(-1))
                off += blk.size
        self._descs, self._pixels = descs, np.concatenate(parts)
        self._values_present = False

    @property
    def blocks(self) -> List[PixlzrBlock]:
        """Vec<PixlzrBlock> view (row-major)."""
        self._materialise_tiles()
        out = []
        c = self._channels
        for d in self._descs:
            n = int(d["w"]) * int(d["h"]) * c
            o = int(d["offset"])
            out.append(PixlzrBlock(self._pixels[o:o + n].reshape(int(d["h"]), int(d["w"]), c),
                                   float(d["value"]) if self._values_present else None))
        return out

    # ---- encode side --------------------------------------------------------------------------------
    def _shrink(self, metric: int, filter_downscale: FilterType, factor: float, flags: int):
        if self._image is None:
            return self._reshrink_blocks(metric, filter_downscale, factor, flags)
        self._encode_source("shrink", lambda img: (img.shrink(self.block_width, self.block_height, metric, factor, int(filter_downscale),
                                                              flags),))

    def _encode_source(self, name: str, encode) -> tuple:
        """Uploads the source image, runs `encode(img)`, which returns a tuple whose first item is a payload, and adopts that
        payload as this Pixlzr's blocks; returns the tuple's other items.  Refused on a decoded or already shrunk Pixlzr."""
        if self._image is None:
            raise ValueError(f"{name} needs the source image (Pixlzr.from_image), not a decoded or already shrunk one")
        with _on_device(self._image, self._ctx()) as img:
            out = encode(img)
            try:
                self._descs, self._pixels = out[0].download()
            finally:
                out[0].free()
        self._values_present = True
        self._image = None
        return out[1:]

    def _reshrink_blocks(self, metric: int, filter_downscale: FilterType, factor: float, flags: int):
        """Shrinks blocks that are no longer windows of the source image (an already shrunk or decoded Pixlzr): the
        reference treats every block as an image of its own (pixlzr.rs:187-205 has no `block_value` check, so
        shrink_directionally re-shrinks reduced blocks).  Blocks of one size are laid side by side into a mosaic whose
        tiles are exactly those blocks, and the mosaic goes through the same device pipeline — the metric, the level
        and the resample of a tile only ever look at that tile."""
        ctx = self._ctx()
        c = self._channels
        descs, pixels = self._descs, self._pixels
        new_descs = descs.copy()
        parts = [None] * len(descs)
        sizes = {}
        for i, d in enumerate(descs):
            sizes.setdefault((int(d["w"]), int(d["h"])), []).append(i)
        for (w, h), idx in sizes.items():
            n = len(idx)
            per_row = max(1, min(n, 16384 // max(w, 1)))
            rows = -(-n // per_row)
            mosaic = np.zeros((rows * h, per_row * w, c), np.uint8)
            for k, i in enumerate(idx):
                o = int(descs[i]["offset"])
                r, q = divmod(k, per_row)
                mosaic[r * h:(r + 1) * h, q * w:(q + 1) * w] = pixels[o:o + w * h * c].reshape(h, w, c)
            if n % per_row:  # the unused tiles of the last mosaic row repeat a real block: same metric domain, results dropped
                o = int(descs[idx[0]]["offset"])
                first = pixels[o:o + w * h * c].reshape(h, w, c)
                for k in range(n, rows * per_row):
                    r, q = divmod(k, per_row)
                    mosaic[r * h:(r + 1) * h, q * w:(q + 1) * w] = first
            img = ctx.image_upload(mosaic)
            try:
                pl = img.shrink(w, h, metric, factor, int(filter_downscale), flags)
                try:
                    md, mp = pl.download()
                finally:
                    pl.free()
            finally:
                img.free()
            for k, i in enumerate(idx):
                dd = md[k]
                o = int(dd["offset"])
                parts[i] = mp[o:o + int(dd["w"]) * int(dd["h"]) * c]
                new_descs[i]["w"], new_descs[i]["h"], new_descs[i]["value"] = dd["w"], dd["h"], dd["value"]
        off = 0
        for i in range(len(new_descs)):
            new_descs[i]["offset"] = off
            off += parts[i].size
        self._descs = new_descs
        self._pixels = np.concatenate(parts) if parts else np.zeros(0, np.uint8)
        self._values_present = True

    def shrink_by(self, filter_downscale: FilterType, factor: float, exact_values: bool = False):
        """Pixlzr::shrink_by (pixlzr.rs:155-185): Oklab-MAD value * factor * 10 -> level -> per-block
        downscale.  Blocks that already carry a value are left alone (:168-170)."""
        if self._image is None and self._values_present:
            return  # every block has block_value.is_some(): the reference clones them unchanged
        self._shrink(N.METRIC_OKLAB_MAD, filter_downscale, factor, N.FLAG_EXACT_VALUES if exact_values else 0)

    def shrink_to_size(self, filter_downscale: FilterType, max_bytes: int, directionally: bool = False,
                       exact_values: bool = False) -> float:
        """EXTENSION (rate control): shrink_by (or shrink_directionally) with the largest factor whose payload has at most
        `max_bytes` bytes; returns that factor (pxz_shrink_to_size).  shrink_by / shrink_directionally with the returned
        factor give the same blocks.  Needs the source image: refused on a decoded or already shrunk Pixlzr."""
        metric = N.METRIC_SOBEL_DIR if directionally else N.METRIC_OKLAB_MAD
        flags = N.FLAG_EXACT_VALUES if exact_values else 0
        k, = self._encode_source("shrink_to_size", lambda img: img.shrink_to_size(self.block_width, self.block_height, metric, max_bytes,
                                                                                  int(filter_downscale), flags))
        return k

    def shrink_to_psnr(self, filter_downscale: FilterType, filter_upscale: FilterType, psnr: float, directionally: bool = False,
                       exact_values: bool = False) -> float:
        """EXTENSION (rate control by error): shrink_by (or shrink_directionally) with the smallest factor whose decode with
        `filter_upscale` reaches `psnr` dB against the source (sse_budget; pxz_shrink_to_error); returns that factor, which is
        also the smallest payload reaching the target.  shrink_by / shrink_directionally with the returned factor give the same
        blocks.  Needs the source image: refused on a decoded or already shrunk Pixlzr."""
        metric = N.METRIC_SOBEL_DIR if directionally else N.METRIC_OKLAB_MAD
        flags = N.FLAG_EXACT_VALUES if exact_values else 0
        k, _ = self._encode_source("shrink_to_psnr", lambda img: img.shrink_to_error(
            self.block_width, self.block_height, metric, sse_budget(psnr, img.w * img.h * img.c), int(filter_downscale),
            int(filter_upscale), flags))
        return k

    def shrink_optimally_to_size(self, filter_downscale: FilterType, filter_upscale: FilterType, max_bytes: int) -> Tuple[int, int]:
        """EXTENSION (optimised encode): each block at its own size, the least error of a decode with `filter_upscale` within
        `max_bytes` payload bytes (pxz_rdo_shrink_to_size); returns (payload bytes, squared error).  Needs the source image:
        refused on a decoded or already shrunk Pixlzr."""
        return self._encode_source("shrink_optimally_to_size", lambda img: img.rdo_shrink_to_size(
            self.block_width, self.block_height, max_bytes, int(filter_downscale), int(filter_upscale)))

    def shrink_optimally_to_psnr(self, filter_downscale: FilterType, filter_upscale: FilterType, psnr: float) -> Tuple[int, int]:
        """EXTENSION (optimised encode): each block at its own size, the fewest payload bytes whose decode with `filter_upscale`
        reaches `psnr` dB against the source (sse_budget; pxz_rdo_shrink_to_error); returns (payload bytes, squared error).
        Needs the source image: refused on a decoded or already shrunk Pixlzr."""
        return self._encode_source("shrink_optimally_to_psnr", lambda img: img.rdo_shrink_to_error(
            self.block_width, self.block_height, sse_budget(psnr, img.w * img.h * img.c), int(filter_downscale), int(filter_upscale)))

    def shrink_directionally(self, filter_downscale: FilterType, factor: float):
        """Pixlzr::shrink_directionally (pixlzr.rs:187-205)."""
        self._shrink(N.METRIC_SOBEL_DIR, filter_downscale, factor, 0)

    def shrink_by_strategy(self, strategy: "Strategy", factor: float):
        """EXTENSION (SURVEY.md §8f N4): shrink_by with the down filter of every block taken from the strategy table
        (strategies.txt / strategies_by_level.txt: the experiment the reference logged but never wired in)."""
        if self._image is None and self._values_present:
            return
        ctx = self._ctx()
        ctx.set_strategy(strategy.down, strategy.up)
        try:
            self._shrink(N.METRIC_OKLAB_MAD, FilterType.Lanczos3, factor, 0)
        finally:
            ctx.set_strategy(None, None)

    def to_image_by_strategy(self, strategy: "Strategy") -> np.ndarray:
        """EXTENSION: to_image with the up filter of every block taken from the strategy table; the bucket comes from
        the value stored with the block, so it also works on a decoded container."""
        if self._image is not None:
            return self._image.copy()
        ctx = self._ctx()
        ctx.set_strategy(strategy.down, strategy.up)
        try:
            return self.to_image(FilterType.Lanczos3)
        finally:
            ctx.set_strategy(None, None)

    def shrink(self, filter_downscale: FilterType, before_average, after_average):
        """Pixlzr::shrink (pixlzr.rs:124-152): `before_average(x, avg)` is applied per pixel and channel, `after_average(x)`
        to the block's mean; blocks that already carry a value are skipped (:135).  The reference takes arbitrary fn
        pointers; the device metric is |x - avg| followed by a linear map, which is what every caller in the reference
        passes (pixlzr.rs:160-162, process/mod.rs:108-110), so the two callables are probed on sample points and
        accepted when they are exactly that; anything else is refused (host-only by nature)."""
        if self._image is None and self._values_present:
            return  # every block has block_value.is_some(): the reference clones them unchanged
        xs = np.array([0.0, 0.25, 1.0, -0.5, 0.7071, 3.5], np.float32)
        avgs = np.array([0.0, 0.5, -0.25, 1.0], np.float32)
        for x in xs:
            for a in avgs:
                if np.float32(before_average(float(x), float(a))) != np.float32(abs(np.float32(x) - np.float32(a))):
                    raise NotImplementedError("before_average is not |x - avg|: arbitrary closures are host-only")
        one = np.float32(after_average(1.0))
        zero = np.float32(after_average(0.0))
        if zero != 0 or any(np.float32(after_average(float(x))) != np.float32(np.float32(x) * one) for x in xs):
            raise NotImplementedError("after_average is not x * c: arbitrary closures are host-only")
        if one == np.float32(1.0):
            self._shrink(N.METRIC_OKLAB_MAD, filter_downscale, 1.0, N.FLAG_AFTER_IDENTITY)
        else:
            # x * c == (x * factor) * 10 needs a factor with that exact product sequence: only c = f32(f * 10) qualifies
            f = np.float32(one / np.float32(10.0))
            if any(np.float32(np.float32(np.float32(x) * f) * np.float32(10.0)) != np.float32(np.float32(x) * one) for x in xs):
                raise NotImplementedError("after_average is not of the form x * factor * 10")
            self._shrink(N.METRIC_OKLAB_MAD, filter_downscale, float(f), 0)

    # ---- decode side --------------------------------------------------------------------------------
    def to_image(self, filter: FilterType) -> np.ndarray:
        """Pixlzr::to_image (pixlzr_image.rs:24-74) = expand + paste, one kernel."""
        if self._image is not None:
            return self._image.copy()  # every block is full size: resize is the identity (block.rs:279-281)
        ctx = self._ctx()
        pl = ctx.payload_upload(self.width, self.height, self.block_width, self.block_height, self._channels,
                                self._descs, self._pixels)
        try:
            return pl.expand(int(filter))
        finally:
            pl.free()

    def to_image_region(self, filter: FilterType, x: int, y: int, w: int, h: int) -> np.ndarray:
        """EXTENSION (random access): to_image(filter)[y:y+h, x:x+w], bit for bit; only the blocks the rectangle touches
        are uploaded and resampled."""
        _check_rect(self.width, self.height, x, y, w, h)
        if self._image is not None:
            return self._image[y:y + h, x:x + w].copy()
        c0, r0, nc, nr = _touched_blocks(self.block_width, self.block_height, x, y, w, h)
        cols = self.block_grid_width()
        idx = ((r0 + np.arange(nr))[:, None] * cols + (c0 + np.arange(nc))[None, :]).reshape(-1)
        descs = self._descs[idx].copy()
        sizes = descs["w"].astype(np.int64) * descs["h"] * self._channels
        descs["offset"] = np.concatenate([[0], np.cumsum(sizes)[:-1]])
        pixels = np.concatenate([self._pixels[o:o + n] for o, n in zip(self._descs["offset"][idx].tolist(), sizes.tolist())])
        x0, y0 = c0 * self.block_width, r0 * self.block_height
        ww = min(self.width, (c0 + nc) * self.block_width) - x0
        wh = min(self.height, (r0 + nr) * self.block_height) - y0
        pl = self._ctx().payload_upload(ww, wh, self.block_width, self.block_height, self._channels, descs, pixels)
        try:
            return pl.expand_region(int(filter), x - x0, y - y0, w, h)
        finally:
            pl.free()

    def expand(self, filter: FilterType) -> "Pixlzr":
        """Pixlzr::expand (pixlzr.rs:77-122): every block resized to its full tile size."""
        out = Pixlzr.from_image(self.to_image(filter), self.block_width, self.block_height, self.ctx)
        out.filter = filter
        out._materialise_tiles()
        if self._values_present:  # resize() resets block_value to None (block.rs:327)
            out._values_present = False
        return out

    # ---- container (host stage) -----------------------------------------------------------------------
    def encode_to_vec(self) -> bytes:
        """Pixlzr::encode_to_vec (encoding/mod.rs:40-89)."""
        self._materialise_tiles()
        vp = None if self._values_present else np.zeros(len(self._descs), np.uint8)
        return N.container_encode(self.width, self.height, self.block_width, self.block_height,
                                  int(self.filter) if self.filter is not None else 0, self._channels, self._descs,
                                  self._pixels, vp)

    @classmethod
    def decode_from_vec(cls, data: bytes) -> "Pixlzr":
        """Pixlzr::decode_from_vec (encoding/mod.rs:95-165)."""
        hdr, descs, pixels = N.container_decode(data)
        p = cls(hdr["w"], hdr["h"], hdr["bw"], hdr["bh"],
                FilterType.from_u8(hdr["filter"]) if hdr["filter"] >= 0 else None)
        p._descs, p._pixels, p._channels = descs, pixels, hdr["channels"]
        p._values_present = True  # decode_block sets Some(value) (encoding/mod.rs:240)
        return p

    # ---- container stage on the device: only the compressed file crosses PCIe ---------------------------
    @staticmethod
    def encode_image_to_vec(image: np.ndarray, block_width: int, block_height: int, filter_downscale: FilterType, factor: float,
                            directionally: bool = False, ctx: Optional[N.Context] = None) -> bytes:
        """from_image + shrink_by (or shrink_directionally) + encode_to_vec in one pass on the device: the per-block QOI
        streams are written by the GPU from the resident payload (pxz_payload_to_container).  Same bytes as the three calls."""
        image = _check_image(image)
        ctx = ctx or default_context()
        img = ctx.image_upload(image)
        try:
            pl = img.shrink(block_width, block_height, N.METRIC_SOBEL_DIR if directionally else N.METRIC_OKLAB_MAD, factor,
                            int(filter_downscale), 0)
            try:
                return pl.to_container(0, True)  # from_image leaves `filter` unset: byte 0
            finally:
                pl.free()
        finally:
            img.free()

    @staticmethod
    def encode_image_to_vec_sized(image: np.ndarray, block_width: int, block_height: int, filter_downscale: FilterType,
                                  max_bytes: int, directionally: bool = False, ctx: Optional[N.Context] = None) -> Tuple[bytes, float]:
        """EXTENSION (rate control): encode_image_to_vec with the largest factor whose payload (not the file) has at most
        `max_bytes` bytes.  Returns (file, factor); encode_image_to_vec with that factor writes the same file."""
        image = _check_image(image)
        ctx = ctx or default_context()
        img = ctx.image_upload(image)
        try:
            pl, k = img.shrink_to_size(block_width, block_height, N.METRIC_SOBEL_DIR if directionally else N.METRIC_OKLAB_MAD,
                                       max_bytes, int(filter_downscale), 0)
            try:
                return pl.to_container(0, True), k
            finally:
                pl.free()
        finally:
            img.free()

    @staticmethod
    def decode_vec_to_image(data: bytes, filter: FilterType, ctx: Optional[N.Context] = None) -> np.ndarray:
        """decode_from_vec + to_image with the QOI streams decoded on the device (pxz_payload_from_container)."""
        ctx = ctx or default_context()
        pl, _ = ctx.payload_from_container(data)
        try:
            return pl.expand(int(filter))
        finally:
            pl.free()

    @staticmethod
    def decode_vec_region_to_image(data, filter: FilterType, x: int, y: int, w: int, h: int,
                                   ctx: Optional[N.Context] = None) -> np.ndarray:
        """EXTENSION (random access): pixels [x, x+w) x [y, y+h) of decode_vec_to_image(data, filter), bit for bit.  Only
        the block rows the rectangle touches are read; the touched blocks are cut out of the file without decoding
        (pxz_container_crop), and only that file crosses PCIe.  `data`: bytes or any buffer, e.g. an mmap of the file."""
        hdr = N.container_header(data)
        _check_rect(hdr["w"], hdr["h"], x, y, w, h)
        c0, r0, nc, nr = _touched_blocks(hdr["bw"], hdr["bh"], x, y, w, h)
        ctx = ctx or default_context()
        pl, _ = ctx.payload_from_container(N.container_crop(data, c0, r0, nc, nr))
        try:
            return pl.expand_region(int(filter), x - c0 * hdr["bw"], y - r0 * hdr["bh"], w, h)
        finally:
            pl.free()

    @classmethod
    def open(cls, path) -> "Pixlzr":
        with open(path, "rb") as f:
            return cls.decode_from_vec(f.read())

    def save(self, path):
        with open(path, "wb") as f:
            f.write(self.encode_to_vec())


# ---- free functions (operations.rs, process/mod.rs) ----------------------------------------------------
def _block_image(block) -> np.ndarray:
    return _check_image(block.data if isinstance(block, PixlzrBlock) else block)


def get_block_variance(block, after=None, exact: bool = True, ctx: Optional[N.Context] = None) -> float:
    """get_block_variance with before = |x - avg| (operations.rs:26-126); `after` is applied on the host."""
    img = _block_image(block)
    ctx = ctx or default_context()
    d = ctx.image_upload(img)
    try:
        vx, _ = d.analyze(img.shape[1], img.shape[0], N.METRIC_OKLAB_MAD, N.FLAG_EXACT_VALUES if exact else 0)
    finally:
        d.free()
    v = np.float32(vx[0])
    return float(after(v)) if after else float(v)


def get_block_variance_directionally(block, ctx: Optional[N.Context] = None) -> Tuple[float, float]:
    """operations.rs:192-259."""
    img = _block_image(block)
    ctx = ctx or default_context()
    d = ctx.image_upload(img)
    try:
        vx, vy = d.analyze(img.shape[1], img.shape[0], N.METRIC_SOBEL_DIR)
    finally:
        d.free()
    return float(vx[0]), float(vy[0])


def reduce_image_section(value: Tuple[float, float], block, filter_downscale: FilterType,
                         ctx: Optional[N.Context] = None) -> PixlzrBlock:
    """operations.rs:140-156 for one block: value -> dims on the host (pxz_reduce_dims, same threshold
    table as the plan kernel), resample on the GPU."""
    img = _block_image(block)
    ctx = ctx or default_context()
    w, h = img.shape[1], img.shape[0]
    nw, nh, stored = N.reduce_dims(value[0], value[1], w, h)
    out = PixlzrBlock(img, None).resize(nw, nh, filter_downscale, ctx)
    out.block_value = stored
    return out


def process_custom(image: np.ndarray, block_width: int, block_height: int, filter_downscale: FilterType,
                   filter_upscale: FilterType, ctx: Optional[N.Context] = None) -> np.ndarray:
    """process_custom (process/mod.rs:71-102) with the closures `process` uses: |x-avg| and identity.
    Output is always RGBA8 (:81-82); RGB inputs get alpha 255 when pasted (copy_from)."""
    image = _check_image(image)
    ctx = ctx or default_context()
    d = ctx.image_upload(image)
    try:
        pl = d.shrink(block_width, block_height, N.METRIC_OKLAB_MAD, 1.0, int(filter_downscale), N.FLAG_AFTER_IDENTITY)
        try:
            out = pl.expand(int(filter_upscale))
        finally:
            pl.free()
    finally:
        d.free()
    if out.shape[2] == 3:
        out = np.concatenate([out, np.full(out.shape[:2] + (1,), 255, np.uint8)], axis=2)
    return out


def process_by_strategy(image: np.ndarray, block_size: int, strategy: Optional[Strategy] = None,
                        ctx: Optional[N.Context] = None) -> np.ndarray:
    """EXTENSION: `process` with a per-block (down, up) filter pair instead of Lanczos3 / Nearest (the experiment of
    strategies.txt; default table: strategies_by_level.txt)."""
    ctx = ctx or default_context()
    strategy = strategy or Strategy.by_level()
    ctx.set_strategy(strategy.down, strategy.up)
    try:
        return process_custom(image, block_size, block_size, FilterType.Lanczos3, FilterType.Lanczos3, ctx)
    finally:
        ctx.set_strategy(None, None)


def process(image: np.ndarray, block_size: int, ctx: Optional[N.Context] = None) -> np.ndarray:
    """process (process/mod.rs:107-121): Lanczos3 down, Nearest up."""
    return process_custom(image, block_size, block_size, FilterType.Lanczos3, FilterType.Nearest, ctx)


def tree_process_custom(image: np.ndarray, threshold: float, block_size: Tuple[int, int], min_block_size: Tuple[int, int],
                        filters: Tuple[FilterType, FilterType], ctx: Optional[N.Context] = None) -> np.ndarray:
    """tree::process_custom (process/tree.rs:23-83) with the closures tree::process uses (|x-avg|, identity).
    Returns RGBA8 like the reference's canvas, except when the block size is already at the minimum: then the input
    comes back unchanged (tree.rs:35-37: `image.clone()`)."""
    image = _check_image(image)
    bw, bh = block_size
    if bw <= max(min_block_size[0], 4) or bh <= max(min_block_size[1], 4):
        return image.copy()
    ctx = ctx or default_context()
    d = ctx.image_upload(image)
    out = ctx.image_alloc(image.shape[1], image.shape[0], image.shape[2])
    try:
        d.tree_process(threshold, bw, bh, min_block_size[0], min_block_size[1], int(filters[0]), int(filters[1]), out)
        res = out.download()
    finally:
        out.free()
        d.free()
    if res.shape[2] == 3:
        res = np.concatenate([res, np.full(res.shape[:2] + (1,), 255, np.uint8)], axis=2)
    return res


def tree_process(image: np.ndarray, block_size: int, threshold: float, ctx: Optional[N.Context] = None) -> np.ndarray:
    """tree::process (process/tree.rs:89-109): Lanczos3 down, Nearest up, minimum block 4."""
    return tree_process_custom(image, threshold, (block_size, block_size), (4, 4), (FilterType.Lanczos3, FilterType.Nearest), ctx)


def format_shrinking_factor(k: float) -> str:
    """The shortest decimal that parse_shrinking_factor reads back to the same f32 (e.g. the factor shrink_to_size chose)."""
    return str(np.float32(k))


def parse_shrinking_factor(s: str) -> float:
    """src/bin/main.rs:47-68: [+|-][1/]D[.D]; unparsable numbers fall back to 1.0."""
    pos, invert, negative = 0, False, False
    if s[pos:].startswith("+"):
        pos += 1
    elif s[pos:].startswith("-"):
        negative = True
        pos += 1
    if s[pos:].startswith("1/"):
        invert = True
        pos += 2
    try:
        body = s[pos:]
        if not body or body.strip() != body or any(ch not in "0123456789.eE+-infa" for ch in body.lower()):
            raise ValueError
        factor = float(np.float32(float(body)))
    except ValueError:
        factor = 1.0
    return (-1.0 if negative else 1.0) * (1.0 / factor if invert else factor)
