"""ctypes binding of libpixlzr_b200.so — the C ABI declared in include/pixlzr_b200.h.

There is no fallback: if the shared library is missing this module raises, and every compute
call returns an error status when no B200 is present.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PXZ_LIB", os.path.join(HERE, "libpixlzr_b200.so"))

OK, E_ARG, E_CUDA, E_OOM, E_NCCL, E_UNSUPPORTED, E_FORMAT = 0, -1, -2, -3, -4, -5, -6
STATUS_NAMES = {0: "PXZ_OK", -1: "PXZ_E_ARG", -2: "PXZ_E_CUDA", -3: "PXZ_E_OOM", -4: "PXZ_E_NCCL",
                -5: "PXZ_E_UNSUPPORTED", -6: "PXZ_E_FORMAT"}
METRIC_OKLAB_MAD, METRIC_SOBEL_DIR = 0, 1
FLAG_AFTER_IDENTITY, FLAG_NORMALISE_GLOBAL, FLAG_EXACT_VALUES = 1, 2, 4
COMM_ID_BYTES = 128
RESIZE_IMAGE_RS, RESIZE_FIR = 0, 1

DESC_DTYPE = np.dtype([("offset", "<u8"), ("value", "<f4"), ("w", "<u2"), ("h", "<u2")])
assert DESC_DTYPE.itemsize == 16

# every symbol include/pixlzr_b200.h declares: name -> (restype, argtypes)
_vp, _u32, _u64, _sz, _i = C.c_void_p, C.c_uint32, C.c_uint64, C.c_size_t, C.c_int
_P = C.POINTER
SYMBOLS = {
    "pxz_abi_version": (_i, []),
    "pxz_device_count": (_i, []),
    "pxz_ctx_create": (_i, [_i, _P(_vp)]),
    "pxz_ctx_create_on_stream": (_i, [_i, _vp, _P(_vp)]),
    "pxz_ctx_destroy": (None, [_vp]),
    "pxz_last_error": (C.c_char_p, [_vp]),
    "pxz_synchronize": (_i, [_vp]),
    "pxz_launch_count": (_u64, [_vp]),
    "pxz_ctx_set_fast_resample": (_i, [_vp, _i]),
    "pxz_ctx_set_resize_semantics": (_i, [_vp, _i]),
    "pxz_strategy_bucket": (_u32, [C.c_float]),
    "pxz_strategy_by_level": (_i, [_vp]),
    "pxz_ctx_set_strategy": (_i, [_vp, _vp]),
    "pxz_profile_enable": (_i, [_vp, _i]),
    "pxz_profile_kernel_name": (C.c_char_p, [_i]),
    "pxz_profile_read": (_i, [_vp, _i, _P(C.c_double), _P(_u64)]),
    "pxz_host_alloc": (_i, [_sz, _P(_vp)]),
    "pxz_host_free": (None, [_vp]),
    "pxz_image_upload": (_i, [_vp, _vp, _u32, _u32, _u32, _sz, _P(_vp)]),
    "pxz_image_alloc": (_i, [_vp, _u32, _u32, _u32, _P(_vp)]),
    "pxz_image_wrap": (_i, [_vp, _vp, _u32, _u32, _u32, _sz, _P(_vp)]),
    "pxz_image_info": (_i, [_vp, _P(_u32), _P(_u32), _P(_u32), _P(_sz), _P(_vp)]),
    "pxz_image_download": (_i, [_vp, _vp, _vp, _sz]),
    "pxz_image_free": (None, [_vp]),
    "pxz_image_alloc_batch": (_i, [_vp, _u32, _u32, _u32, _u32, _P(_vp)]),
    "pxz_image_upload_batch": (_i, [_vp, _vp, _u32, _u32, _u32, _sz, _u32, _P(_vp)]),
    "pxz_image_wrap_batch": (_i, [_vp, _vp, _u32, _u32, _u32, _sz, _u32, _P(_vp)]),
    "pxz_image_batch_count": (_u32, [_vp]),
    "pxz_shrink_batch": (_i, [_vp, _vp, _u32, _u32, _i, C.c_float, _i, _u32, _P(_vp)]),
    "pxz_expand_batch": (_i, [_vp, _vp, _i, _vp]),
    "pxz_payload_upload_batch": (_i, [_vp, _u32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _u64, _P(_vp)]),
    "pxz_payload_batch_count": (_u32, [_vp]),
    "pxz_grid": (_i, [_u32, _u32, _u32, _u32, _P(_u32), _P(_u32)]),
    "pxz_analyze": (_i, [_vp, _vp, _u32, _u32, _i, _u32, _vp, _vp]),
    "pxz_shrink": (_i, [_vp, _vp, _u32, _u32, _i, C.c_float, _i, _u32, _P(_vp)]),
    "pxz_shrink_to_size": (_i, [_vp, _vp, _u32, _u32, _i, _u64, _i, _u32, _P(C.c_float), _P(_vp)]),
    "pxz_reduce_dims": (_i, [C.c_float, C.c_float, _u32, _u32, _P(_u32), _P(_u32), _P(C.c_float)]),
    "pxz_resample_table": (C.c_int32, [_u32, _u32, _i, _vp, _vp, _vp, _u32]),
    "pxz_payload_info": (_i, [_vp, _vp] + [_P(_u32)] * 7 + [_P(_u64)]),
    "pxz_payload_download": (_i, [_vp, _vp, _vp, _vp]),
    "pxz_payload_upload": (_i, [_vp, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _u64, _P(_vp)]),
    "pxz_payload_free": (None, [_vp]),
    "pxz_expand": (_i, [_vp, _vp, _i, _vp, _sz]),
    "pxz_expand_to_image": (_i, [_vp, _vp, _i, _vp]),
    "pxz_tree_process": (_i, [_vp, _vp, C.c_float, _u32, _u32, _u32, _u32, _i, _i, _vp]),
    "pxz_comm_unique_id": (_i, [_vp]),
    "pxz_comm_init": (_i, [_vp, _i, _i, _vp]),
    "pxz_comm_destroy": (None, [_vp]),
    "pxz_comm_join_empty": (_i, [_vp]),
    "pxz_container_bound": (C.c_int64, [_u32, _u32, _u32, _u32, _u32, _u64]),
    "pxz_container_encode": (C.c_int64, [_u32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _sz, _i]),
    "pxz_payload_to_container": (_i, [_vp, _vp, _u32, _i, _vp, _sz, _P(_u64)]),
    "pxz_payload_from_container": (_i, [_vp, _vp, _sz, _P(C.c_int32), _P(_vp)]),
    "pxz_container_decode": (_i, [_vp, _sz, _P(_u32), _P(_u32), _P(_u32), _P(_u32), _P(C.c_int32), _P(_u32),
                                  _P(_u64), _vp, _vp]),
    "pxz_payload_window": (_i, [_vp, _vp, _u32, _u32, _u32, _u32, _P(_vp)]),
    "pxz_expand_region": (_i, [_vp, _vp, _i, _u32, _u32, _u32, _u32, _vp]),
    "pxz_container_header": (_i, [_vp, _sz, _P(_u32), _P(_u32), _P(_u32), _P(_u32), _P(C.c_int32)]),
    "pxz_container_crop": (C.c_int64, [_vp, _sz, _u32, _u32, _u32, _u32, _vp, _sz]),
    "pxz_image_error": (_i, [_vp, _vp, _vp, _u32, _u32, _vp, _vp, _P(_u64)]),
    "pxz_strategy_measure": (_i, [_vp, _vp, _u32, _u32, _i, C.c_float, _u32, _vp, _vp]),
    "pxz_strategy_choose": (_i, [_vp, _vp, _vp, _vp]),
    "pxz_rd_curve": (_i, [_vp, _vp, _u32, _u32, _i, _i, _i, _u32, _vp, _vp, _vp, _sz, _P(_sz)]),
    "pxz_shrink_to_error": (_i, [_vp, _vp, _u32, _u32, _i, _u64, _i, _i, _u32, _P(C.c_float), _P(_u64), _P(_vp)]),
    "pxz_rdo_curve": (_i, [_vp, _vp, _u32, _u32, _i, _i, _vp, _vp, _sz, _P(_sz)]),
    "pxz_rdo_shrink_to_size": (_i, [_vp, _vp, _u32, _u32, _u64, _i, _i, _P(_u64), _P(_u64), _P(_vp)]),
    "pxz_rdo_shrink_to_error": (_i, [_vp, _vp, _u32, _u32, _u64, _i, _i, _P(_u64), _P(_u64), _P(_vp)]),
}


class PixlzrError(RuntimeError):
    def __init__(self, status: int, message: str = ""):
        self.status = status
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {message}")


_lib = None


def lib():
    """Loads libpixlzr_b200.so; raises if it has not been built (python pixlzr-rust_b200/build.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python pixlzr-rust_b200/build.py` "
                "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        if L.pxz_abi_version() != 1:
            raise ImportError("libpixlzr_b200.so ABI version mismatch")
        _lib = L
    return _lib


def ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    return a


STRATEGY_BUCKETS = 65


def strategy_bucket(value: float) -> int:
    return int(lib().pxz_strategy_bucket(float(value)))


def strategy_by_level():
    """(down, up) uint8[65]: the table of strategies_by_level.txt (pxz_strategy_by_level)."""
    buf = np.zeros(2 * STRATEGY_BUCKETS, np.uint8)
    rc = lib().pxz_strategy_by_level(buf.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise RuntimeError(f"pxz_strategy_by_level failed ({rc})")
    return buf[:STRATEGY_BUCKETS].copy(), buf[STRATEGY_BUCKETS:].copy()


FILTER_PAIRS = 25  # pair index = down * 5 + up


def strategy_choose(sse: np.ndarray, blocks: np.ndarray, base=None):
    """(down, up) uint8[65]: per bucket the (down, up) pair of least summed error in a strategy_measure report (summed over
    any number of images); ties keep base's pair, else the lowest pair index; empty buckets keep base's pair.  base: (down,
    up) or None for strategy_by_level (pxz_strategy_choose)."""
    sse = np.ascontiguousarray(sse, np.uint64)
    blocks = np.ascontiguousarray(blocks, np.uint32)
    if sse.size != STRATEGY_BUCKETS * FILTER_PAIRS or blocks.size != STRATEGY_BUCKETS:
        raise ValueError(f"a report has {STRATEGY_BUCKETS} x {FILTER_PAIRS} sums and {STRATEGY_BUCKETS} counts")
    basebuf = None
    if base is not None:
        basebuf = np.concatenate([np.asarray(base[0], np.uint8).reshape(-1), np.asarray(base[1], np.uint8).reshape(-1)])
        if basebuf.size != 2 * STRATEGY_BUCKETS:
            raise ValueError(f"a strategy has {STRATEGY_BUCKETS} entries per direction")
    out = np.zeros(2 * STRATEGY_BUCKETS, np.uint8)
    st = lib().pxz_strategy_choose(ptr(sse), ptr(blocks), ptr(basebuf), ptr(out))
    if st != OK:
        raise PixlzrError(st, "pxz_strategy_choose")
    return out[:STRATEGY_BUCKETS].copy(), out[STRATEGY_BUCKETS:].copy()


class PinnedBuffer:
    """Page-locked host bytes (pxz_host_alloc) as a numpy uint8 array; freed with the object."""

    def __init__(self, nbytes: int):
        self._p = C.c_void_p()
        st = lib().pxz_host_alloc(max(1, int(nbytes)), C.byref(self._p))
        if st != OK:
            self._p = C.c_void_p()
            raise PixlzrError(st, "pxz_host_alloc")
        self.array = np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_uint8)), shape=(max(1, int(nbytes)),))

    def __del__(self):
        if getattr(self, "_p", None) is not None and self._p.value:
            self.array = None
            lib().pxz_host_free(self._p)
            self._p = C.c_void_p()


class Context:
    """One device + one stream (pxz_ctx).  Not thread-safe; use one per thread."""
    _staging: "PinnedBuffer | None" = None

    def staging(self, nbytes: int) -> np.ndarray:
        """A pinned scratch array of at least `nbytes` owned by the context (grows, never shrinks)."""
        if self._staging is None or self._staging.array.size < nbytes:
            self._staging = None
            self._staging = PinnedBuffer(nbytes)
        return self._staging.array

    def __init__(self, device: int = 0, cuda_stream: int | None = None):
        self._h = C.c_void_p()
        L = lib()
        if cuda_stream is None:
            st = L.pxz_ctx_create(device, C.byref(self._h))
        else:
            st = L.pxz_ctx_create_on_stream(device, C.c_void_p(cuda_stream), C.byref(self._h))
        if st != OK:
            self._h = C.c_void_p()
            raise PixlzrError(st, "cannot create a context: no usable sm_100 (B200) device"
                              if st == E_CUDA else "pxz_ctx_create")
        self.device = device

    @property
    def handle(self):
        return self._h

    def check(self, st: int):
        if st != OK:
            raise PixlzrError(st, lib().pxz_last_error(self._h).decode(errors="replace"))

    def synchronize(self):
        self.check(lib().pxz_synchronize(self._h))

    def launch_count(self) -> int:
        return int(lib().pxz_launch_count(self._h))

    def set_fast_resample(self, on: bool = True):
        """Fused multiply-add in the RGBA resample kernels: pixels within +-1 LSB instead of bit-exact."""
        self.check(lib().pxz_ctx_set_fast_resample(self._h, int(on)))

    def set_strategy(self, down=None, up=None):
        """Per-block filter pairs (pxz_ctx_set_strategy): `down` / `up` are 65 filter ids indexed by
        strategy_bucket(block value); None removes the strategy."""
        if down is None or up is None:
            self.check(lib().pxz_ctx_set_strategy(self._h, None))
            return
        buf = np.concatenate([np.asarray(down, np.uint8).reshape(-1), np.asarray(up, np.uint8).reshape(-1)])
        if buf.size != 2 * STRATEGY_BUCKETS:
            raise ValueError(f"a strategy has {STRATEGY_BUCKETS} entries per direction")
        self.check(lib().pxz_ctx_set_strategy(self._h, buf.ctypes.data_as(C.c_void_p)))

    def profile_enable(self, on: bool = True):
        self.check(lib().pxz_profile_enable(self._h, int(on)))

    def profile_read(self) -> dict:
        """{kernel name: (total ms, launches)} since profiling was enabled (synchronises)."""
        out, i = {}, 0
        while True:
            name = lib().pxz_profile_kernel_name(i)
            if name is None:
                break
            ms, n = C.c_double(), C.c_uint64()
            self.check(lib().pxz_profile_read(self._h, i, C.byref(ms), C.byref(n)))
            out[name.decode()] = (ms.value, n.value)
            i += 1
        return out

    def set_resize_semantics(self, semantics: int):
        """RESIZE_IMAGE_RS (default, pinned by the reference's fixtures) or RESIZE_FIR (the reference's default cargo
        feature; parity unpinned)."""
        self.check(lib().pxz_ctx_set_resize_semantics(self._h, int(semantics)))

    def comm_join_empty(self):
        """The exchange of one PXZ_FLAG_NORMALISE_GLOBAL shrink for a rank whose shard has no block rows."""
        self.check(lib().pxz_comm_join_empty(self._h))

    def comm_init(self, nranks: int, rank: int, comm_id: bytes):
        """Joins the NCCL communicator used by PXZ_FLAG_NORMALISE_GLOBAL (all ranks must call this)."""
        assert len(comm_id) == COMM_ID_BYTES
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(comm_id)
        self.check(lib().pxz_comm_init(self._h, nranks, rank, buf))

    def close(self):
        if self._h:
            lib().pxz_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- images -------------------------------------------------------------------------------
    def image_upload(self, img: np.ndarray) -> "Image":
        assert img.dtype == np.uint8 and img.ndim == 3 and img.shape[2] in (3, 4)
        assert img.strides[2] == 1 and img.strides[1] == img.shape[2], "pixels must be interleaved"
        h = C.c_void_p()
        self.check(lib().pxz_image_upload(self._h, ptr(img), img.shape[1], img.shape[0], img.shape[2],
                                          img.strides[0], C.byref(h)))
        return Image(self, h, img.shape[1], img.shape[0], img.shape[2])

    def image_alloc(self, w: int, h: int, c: int) -> "Image":
        hd = C.c_void_p()
        self.check(lib().pxz_image_alloc(self._h, w, h, c, C.byref(hd)))
        return Image(self, hd, w, h, c)

    def image_wrap(self, device_ptr: int, w: int, h: int, c: int, pitch: int) -> "Image":
        hd = C.c_void_p()
        self.check(lib().pxz_image_wrap(self._h, C.c_void_p(device_ptr), w, h, c, pitch, C.byref(hd)))
        return Image(self, hd, w, h, c)

    # ---- batches: n images of one size stacked in one allocation (include/pixlzr_b200.h "batches of images") ----
    def image_upload_batch(self, imgs: np.ndarray) -> "Image":
        """imgs: uint8 [n, h, w, c], C-contiguous."""
        assert imgs.dtype == np.uint8 and imgs.ndim == 4 and imgs.shape[3] in (3, 4) and imgs.flags.c_contiguous
        n, h, w, c = imgs.shape
        hd = C.c_void_p()
        self.check(lib().pxz_image_upload_batch(self._h, ptr(imgs), w, h, c, imgs.strides[1], n, C.byref(hd)))
        return Image(self, hd, w, h, c, n)

    def image_alloc_batch(self, w: int, h: int, c: int, n: int) -> "Image":
        hd = C.c_void_p()
        self.check(lib().pxz_image_alloc_batch(self._h, w, h, c, n, C.byref(hd)))
        return Image(self, hd, w, h, c, n)

    def image_wrap_batch(self, device_ptr: int, w: int, h: int, c: int, pitch: int, n: int) -> "Image":
        hd = C.c_void_p()
        self.check(lib().pxz_image_wrap_batch(self._h, C.c_void_p(device_ptr), w, h, c, pitch, n, C.byref(hd)))
        return Image(self, hd, w, h, c, n)

    def payload_upload_batch(self, w, h, bw, bh, c, n, descs: np.ndarray, pixels: np.ndarray) -> "Payload":
        assert descs.dtype == DESC_DTYPE and pixels.dtype == np.uint8
        descs = np.ascontiguousarray(descs)
        pixels = np.ascontiguousarray(pixels)
        hd = C.c_void_p()
        self.check(lib().pxz_payload_upload_batch(self._h, w, h, bw, bh, c, n, ptr(descs), ptr(pixels), pixels.size, C.byref(hd)))
        return Payload(self, hd)

    # ---- payload ------------------------------------------------------------------------------
    def payload_upload(self, w, h, bw, bh, c, descs: np.ndarray, pixels: np.ndarray) -> "Payload":
        assert descs.dtype == DESC_DTYPE and pixels.dtype == np.uint8
        descs = np.ascontiguousarray(descs)
        pixels = np.ascontiguousarray(pixels)
        hd = C.c_void_p()
        self.check(lib().pxz_payload_upload(self._h, w, h, bw, bh, c, ptr(descs), ptr(pixels), pixels.size, C.byref(hd)))
        return Payload(self, hd)


    def payload_from_container(self, data: bytes):
        """(Payload, filter byte or -1): a .pxlzr file decoded on the device (pxz_payload_from_container)."""
        buf = np.frombuffer(data, np.uint8)
        hd, filt = C.c_void_p(), C.c_int32(-1)
        self.check(lib().pxz_payload_from_container(self._h, ptr(buf), len(data), C.byref(filt), C.byref(hd)))
        return Payload(self, hd), int(filt.value)


class Image:
    def __init__(self, ctx: Context, handle, w, h, c, n: int = 1):
        self.ctx, self._h, self.w, self.h, self.c, self.n = ctx, handle, w, h, c, n

    @property
    def handle(self):
        return self._h

    def info(self):
        w, h, c, pitch, p = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_size_t(), C.c_void_p()
        self.ctx.check(lib().pxz_image_info(self._h, C.byref(w), C.byref(h), C.byref(c), C.byref(pitch), C.byref(p)))
        return dict(w=w.value, h=h.value, channels=c.value, pitch=pitch.value, device_ptr=p.value)

    def download(self) -> np.ndarray:
        """[h, w, c], or [n, h, w, c] for a batch."""
        out = np.empty((self.n * self.h, self.w, self.c), np.uint8)
        self.ctx.check(lib().pxz_image_download(self.ctx.handle, self._h, ptr(out), out.strides[0]))
        return out if self.n == 1 else out.reshape(self.n, self.h, self.w, self.c)

    def analyze(self, bw: int, bh: int, metric: int, flags: int = 0):
        cols, rows = grid(self.w, self.h, bw, bh)
        vx = np.empty(cols * rows * self.n, np.float32)  # a batch: image after image
        vy = np.empty(cols * rows * self.n, np.float32)
        self.ctx.check(lib().pxz_analyze(self.ctx.handle, self._h, bw, bh, metric, flags, ptr(vx), ptr(vy)))
        return vx, vy

    def shrink(self, bw: int, bh: int, metric: int, factor: float, filter_down: int, flags: int = 0) -> "Payload":
        h = C.c_void_p()
        self.ctx.check(lib().pxz_shrink(self.ctx.handle, self._h, bw, bh, metric, factor, int(filter_down), flags,
                                        C.byref(h)))
        return Payload(self.ctx, h)

    def shrink_to_size(self, bw: int, bh: int, metric: int, max_bytes: int, filter_down: int, flags: int = 0):
        """(Payload, k): the payload of shrink(..., k, ...) for the largest factor k whose payload has at most `max_bytes`
        bytes (pxz_shrink_to_size; k = FLT_MAX when even that fits)."""
        h, k = C.c_void_p(), C.c_float()
        self.ctx.check(lib().pxz_shrink_to_size(self.ctx.handle, self._h, bw, bh, metric, int(max_bytes), int(filter_down), flags,
                                                C.byref(k), C.byref(h)))
        return Payload(self.ctx, h), float(k.value)

    def error(self, other: "Image", bw: int, bh: int):
        """(block_sse uint64 [rows, cols], block_max uint8 [rows, cols], total_sse): the squared error and the largest
        difference of every tile of the (bw, bh) grid between this image and `other` (pxz_image_error; exact)."""
        cols, rows = grid(self.w, self.h, bw, bh)
        sse = np.empty((rows, cols), np.uint64)
        mx = np.empty((rows, cols), np.uint8)
        total = C.c_uint64()
        self.ctx.check(lib().pxz_image_error(self.ctx.handle, self._h, other.handle, bw, bh, ptr(sse), ptr(mx), C.byref(total)))
        return sse, mx, int(total.value)

    def strategy_measure(self, bw: int, bh: int, metric: int, factor: float, flags: int = 0):
        """(sse uint64 [65, 25], blocks uint32 [65]): for every (down, up) pair (index down * 5 + up) the error of
        expand(shrink(self, ..., down, flags), up) against this image, summed per strategy bucket of the stored block
        values, and the block count per bucket (pxz_strategy_measure)."""
        sse = np.zeros((STRATEGY_BUCKETS, FILTER_PAIRS), np.uint64)
        blocks = np.zeros(STRATEGY_BUCKETS, np.uint32)
        self.ctx.check(lib().pxz_strategy_measure(self.ctx.handle, self._h, bw, bh, metric, factor, flags, ptr(sse), ptr(blocks)))
        return sse, blocks

    def rd_curve(self, bw: int, bh: int, metric: int, filter_down: int, filter_up: int, flags: int = 0):
        """(factor float32 [n], bytes uint64 [n], sse uint64 [n]): every distinct payload shrink(bw, bh, metric, k, filter_down,
        flags) gives over the finite k > 0, at the smallest k giving it, with the squared error of its decode with filter_up
        against this image (pxz_rd_curve)."""
        cap = rd_curve_bound(self.w, self.h, bw, bh, metric)
        factor = np.empty(cap, np.float32)
        nbytes = np.empty(cap, np.uint64)
        sse = np.empty(cap, np.uint64)
        n = C.c_size_t()
        self.ctx.check(lib().pxz_rd_curve(self.ctx.handle, self._h, bw, bh, metric, int(filter_down), int(filter_up), flags, ptr(factor),
                                          ptr(nbytes), ptr(sse), cap, C.byref(n)))
        return factor[:n.value].copy(), nbytes[:n.value].copy(), sse[:n.value].copy()

    def shrink_to_error(self, bw: int, bh: int, metric: int, max_sse: int, filter_down: int, filter_up: int, flags: int = 0):
        """(Payload, k, sse): the payload of shrink(..., k, ...) for the smallest factor k whose decode with filter_up has a
        squared error of at most `max_sse` against this image, and that error (pxz_shrink_to_error)."""
        h, k, sse = C.c_void_p(), C.c_float(), C.c_uint64()
        self.ctx.check(lib().pxz_shrink_to_error(self.ctx.handle, self._h, bw, bh, metric, int(max_sse), int(filter_down), int(filter_up),
                                                 flags, C.byref(k), C.byref(sse), C.byref(h)))
        return Payload(self.ctx, h), float(k.value), int(sse.value)

    def rdo_curve(self, bw: int, bh: int, filter_down: int, filter_up: int):
        """(bytes uint64 [n], sse uint64 [n]): the rate-distortion optimised curve of this image, every block free to take the
        dims of any level pair, decoded with filter_up (pxz_rdo_curve)."""
        cap = rdo_curve_bound(self.w, self.h, bw, bh)
        nbytes = np.empty(cap, np.uint64)
        sse = np.empty(cap, np.uint64)
        n = C.c_size_t()
        self.ctx.check(lib().pxz_rdo_curve(self.ctx.handle, self._h, bw, bh, int(filter_down), int(filter_up), ptr(nbytes), ptr(sse), cap,
                                           C.byref(n)))
        return nbytes[:n.value].copy(), sse[:n.value].copy()

    def rdo_shrink_to_size(self, bw: int, bh: int, max_bytes: int, filter_down: int, filter_up: int):
        """(Payload, bytes, sse): the payload of the last optimised curve point with at most `max_bytes` payload bytes, its bytes
        and the squared error of its decode with filter_up (pxz_rdo_shrink_to_size)."""
        h, nbytes, sse = C.c_void_p(), C.c_uint64(), C.c_uint64()
        self.ctx.check(lib().pxz_rdo_shrink_to_size(self.ctx.handle, self._h, bw, bh, int(max_bytes), int(filter_down), int(filter_up),
                                                    C.byref(nbytes), C.byref(sse), C.byref(h)))
        return Payload(self.ctx, h), int(nbytes.value), int(sse.value)

    def rdo_shrink_to_error(self, bw: int, bh: int, max_sse: int, filter_down: int, filter_up: int):
        """(Payload, bytes, sse): the payload of the first optimised curve point whose decode with filter_up has a squared
        error of at most `max_sse`, its bytes and that error (pxz_rdo_shrink_to_error)."""
        h, nbytes, sse = C.c_void_p(), C.c_uint64(), C.c_uint64()
        self.ctx.check(lib().pxz_rdo_shrink_to_error(self.ctx.handle, self._h, bw, bh, int(max_sse), int(filter_down), int(filter_up),
                                                     C.byref(nbytes), C.byref(sse), C.byref(h)))
        return Payload(self.ctx, h), int(nbytes.value), int(sse.value)

    def tree_process(self, threshold: float, bw: int, bh: int, min_bw: int, min_bh: int, filter_down: int, filter_up: int,
                     out: "Image"):
        self.ctx.check(lib().pxz_tree_process(self.ctx.handle, self._h, threshold, bw, bh, min_bw, min_bh, int(filter_down),
                                              int(filter_up), out.handle))

    def free(self):
        if self._h:
            if self.ctx.handle:  # see Payload.free
                lib().pxz_image_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Payload:
    def __init__(self, ctx: Context, handle):
        self.ctx, self._h = ctx, handle

    @property
    def handle(self):
        return self._h

    def to_container_into(self, out: np.ndarray, filter_byte: int = 0, values_present: bool = True) -> int:
        """to_container into a caller-owned uint8 buffer (pinned memory makes the copy run at PCIe speed); returns the size."""
        assert out.dtype == np.uint8 and out.flags.c_contiguous
        n = C.c_uint64()
        self.ctx.check(lib().pxz_payload_to_container(self.ctx.handle, self._h, int(filter_byte), int(values_present), ptr(out), out.size,
                                                      C.byref(n)))
        return int(n.value)

    def to_container(self, filter_byte: int = 0, values_present: bool = True) -> bytes:
        """The .pxlzr file of this payload, QOI streams written on the device (pxz_payload_to_container)."""
        i = self.info()
        cap = lib().pxz_container_bound(i["w"], i["h"], i["bw"], i["bh"], i["channels"], i["bytes"])
        if cap < 0:
            raise PixlzrError(int(cap), "pxz_container_bound")
        out = self.ctx.staging(cap) if cap <= (1 << 30) else np.empty(cap, np.uint8)  # pinned: the file comes back at PCIe speed
        n = C.c_uint64()
        self.ctx.check(lib().pxz_payload_to_container(self.ctx.handle, self._h, int(filter_byte), int(values_present), ptr(out), out.size,
                                                      C.byref(n)))
        return out[:n.value].tobytes()

    def info(self):
        v = [C.c_uint32() for _ in range(7)]
        b = C.c_uint64()
        self.ctx.check(lib().pxz_payload_info(self.ctx.handle, self._h, *[C.byref(x) for x in v], C.byref(b)))
        keys = ["w", "h", "bw", "bh", "cols", "rows", "channels"]
        d = {k: x.value for k, x in zip(keys, v)}
        d["bytes"] = b.value
        d["images"] = int(lib().pxz_payload_batch_count(self._h))  # cols / rows describe ONE image
        return d

    def download(self):
        i = self.info()
        descs = np.empty(i["cols"] * i["rows"] * i["images"], DESC_DTYPE)
        pixels = np.empty(max(1, i["bytes"]), np.uint8)
        self.ctx.check(lib().pxz_payload_download(self.ctx.handle, self._h, ptr(descs), ptr(pixels)))
        return descs, pixels[:i["bytes"]]

    def download_into(self, descs: np.ndarray, pixels: np.ndarray) -> int:
        """Like download(), into caller-provided (e.g. pinned) buffers; returns the payload byte count."""
        i = self.info()
        assert descs.dtype == DESC_DTYPE and descs.size >= i["cols"] * i["rows"] * i["images"] and pixels.size >= i["bytes"]
        self.ctx.check(lib().pxz_payload_download(self.ctx.handle, self._h, ptr(descs), ptr(pixels)))
        return i["bytes"]

    def expand_into(self, filter_up: int, out: np.ndarray):
        self.ctx.check(lib().pxz_expand(self.ctx.handle, self._h, int(filter_up), ptr(out), out.strides[0]))

    def expand(self, filter_up: int) -> np.ndarray:
        i = self.info()
        out = np.empty((i["images"] * i["h"], i["w"], i["channels"]), np.uint8)
        self.ctx.check(lib().pxz_expand(self.ctx.handle, self._h, int(filter_up), ptr(out), out.strides[0]))
        return out if i["images"] == 1 else out.reshape(i["images"], i["h"], i["w"], i["channels"])

    def expand_to_image(self, filter_up: int, out: Image):
        self.ctx.check(lib().pxz_expand_to_image(self.ctx.handle, self._h, int(filter_up), out.handle))

    def error(self, source: Image, filter_up: int):
        """Image.error of the decode (expand_to_image into a scratch image) against `source`, on this payload's block grid."""
        i = self.info()
        img = self.ctx.image_alloc(i["w"], i["h"], i["channels"])
        try:
            self.expand_to_image(filter_up, img)
            return img.error(source, i["bw"], i["bh"])
        finally:
            img.free()

    # ---- random access (extension) -----------------------------------------------------------------------
    def window(self, c0: int, r0: int, nc: int, nr: int) -> "Payload":
        """The blocks of columns [c0, c0+nc) x rows [r0, r0+nr) as a payload of their own (pxz_payload_window)."""
        h = C.c_void_p()
        self.ctx.check(lib().pxz_payload_window(self.ctx.handle, self._h, c0, r0, nc, nr, C.byref(h)))
        return Payload(self.ctx, h)

    def expand_region_to_image(self, filter_up: int, x: int, y: int, w: int, h: int, out: Image):
        """Pixels [x, x+w) x [y, y+h) of the decoded image into `out` (w x h), e.g. an image_wrap'ped torch tensor."""
        self.ctx.check(lib().pxz_expand_region(self.ctx.handle, self._h, int(filter_up), x, y, w, h, out.handle))

    def expand_region(self, filter_up: int, x: int, y: int, w: int, h: int) -> np.ndarray:
        """[h, w, c]: pixels [x, x+w) x [y, y+h) of expand(filter_up), resampling only the blocks they touch."""
        img = self.ctx.image_alloc(w, h, self.info()["channels"])  # an empty rectangle fails here with PXZ_E_ARG
        try:
            self.expand_region_to_image(filter_up, x, y, w, h, img)
            return img.download()
        finally:
            img.free()

    def free(self):
        if self._h:
            # pxz_payload_free returns the buffers to the context (its cache, its stream).  Once the context is closed — or
            # finalised first, as the garbage collector may do with a cycle holding both — the handle is only dropped: its
            # device memory stays allocated until the process ends.
            if self.ctx.handle:
                lib().pxz_payload_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def grid(w, h, bw, bh):
    c, r = C.c_uint32(), C.c_uint32()
    st = lib().pxz_grid(w, h, bw, bh, C.byref(c), C.byref(r))
    if st != OK:
        raise PixlzrError(st, "pxz_grid")
    return c.value, r.value


def rd_curve_bound(w: int, h: int, bw: int, bh: int, metric: int) -> int:
    """Most points pxz_rd_curve can return: 1 + blocks * (ceil(log2 bw) + ceil(log2 bh)), Oklab-MAD ceil(log2 max(bw, bh)) (a
    block's dims change at most once per level it can step through)."""
    if w <= 0 or h <= 0 or bw <= 0 or bh <= 0:
        raise ValueError("image and block sizes must be positive")
    lx, ly = (bw - 1).bit_length(), (bh - 1).bit_length()
    steps = lx + ly if metric == METRIC_SOBEL_DIR else max(lx, ly)
    return 1 + -(-w // bw) * -(-h // bh) * steps


def rdo_curve_bound(w: int, h: int, bw: int, bh: int) -> int:
    """Most points pxz_rdo_curve can return: 1 + blocks * ((1 + ceil(log2 bw)) * (1 + ceil(log2 bh)) - 1) (a block has at most
    one hull segment per candidate size after its first)."""
    if w <= 0 or h <= 0 or bw <= 0 or bh <= 0:
        raise ValueError("image and block sizes must be positive")
    lx, ly = (bw - 1).bit_length(), (bh - 1).bit_length()
    return 1 + -(-w // bw) * -(-h // bh) * ((1 + lx) * (1 + ly) - 1)


def reduce_dims(v0: float, v1: float, w: int, h: int):
    ow, oh, st = C.c_uint32(), C.c_uint32(), C.c_float()
    rc = lib().pxz_reduce_dims(v0, v1, w, h, C.byref(ow), C.byref(oh), C.byref(st))
    if rc != OK:
        raise PixlzrError(rc, "pxz_reduce_dims")
    return ow.value, oh.value, st.value


def comm_unique_id() -> bytes:
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    st = lib().pxz_comm_unique_id(buf)
    if st != OK:
        raise PixlzrError(st, "pxz_comm_unique_id (is libnccl.so.2 loadable?)")
    return bytes(buf)


def resample_table(n_in: int, n_out: int, filt: int):
    """(left, count, weights[n_out, taps]) of one resample axis as the kernels apply it."""
    max_taps = max(1, n_in)
    left = np.zeros(n_out, np.uint32)
    count = np.zeros(n_out, np.uint32)
    w = np.zeros((n_out, max_taps), np.float32)
    rc = lib().pxz_resample_table(n_in, n_out, int(filt), ptr(left), ptr(count), ptr(w), max_taps)
    if rc < 0 or rc > max_taps:
        raise PixlzrError(rc if rc < 0 else E_ARG, "pxz_resample_table")
    return left, count, w[:, :rc].copy()


def device_count() -> int:
    return int(lib().pxz_device_count())


def container_encode(w, h, bw, bh, filter_byte, channels, descs, pixels, value_present=None, nthreads=0) -> bytes:
    descs = np.ascontiguousarray(descs)
    pixels = np.ascontiguousarray(pixels)
    cap = lib().pxz_container_bound(w, h, bw, bh, channels, pixels.size)
    if cap < 0:
        raise PixlzrError(int(cap), "pxz_container_bound")
    out = np.empty(cap, np.uint8)
    if nthreads <= 0:
        nthreads = os.cpu_count() or 1
    vp = None if value_present is None else np.ascontiguousarray(value_present, dtype=np.uint8)
    n = lib().pxz_container_encode(w, h, bw, bh, filter_byte, channels, ptr(descs), ptr(pixels), ptr(vp), ptr(out),
                                   cap, nthreads)
    if n < 0:
        raise PixlzrError(int(n), "pxz_container_encode")
    return out[:n].tobytes()


def container_decode(data: bytes):
    buf = np.frombuffer(data, np.uint8)
    w, h, bw, bh, ch = (C.c_uint32() for _ in range(5))
    filt, nbytes = C.c_int32(), C.c_uint64()
    args = [ptr(buf), len(data), C.byref(w), C.byref(h), C.byref(bw), C.byref(bh), C.byref(filt), C.byref(ch),
            C.byref(nbytes)]
    st = lib().pxz_container_decode(*args, None, None)
    if st != OK:
        raise PixlzrError(st, "malformed .pxlzr container")
    cols = int(np.ceil(np.float32(w.value) / np.float32(bw.value)))
    rows = int(np.ceil(np.float32(h.value) / np.float32(bh.value)))
    descs = np.zeros(cols * rows, DESC_DTYPE)
    pixels = np.zeros(max(1, nbytes.value), np.uint8)
    st = lib().pxz_container_decode(*args, ptr(descs), ptr(pixels))
    if st != OK:
        raise PixlzrError(st, "malformed .pxlzr container")
    hdr = dict(w=w.value, h=h.value, bw=bw.value, bh=bh.value, filter=filt.value, channels=ch.value)
    return hdr, descs, pixels[:nbytes.value]


def container_header(data) -> dict:
    """{w, h, bw, bh, filter} of a .pxlzr file without reading its blocks (pxz_container_header).  `data`: any buffer
    (bytes, mmap, ...); only the header and the line table are read."""
    buf = np.frombuffer(data, np.uint8)
    w, h, bw, bh = (C.c_uint32() for _ in range(4))
    filt = C.c_int32()
    st = lib().pxz_container_header(ptr(buf), buf.size, C.byref(w), C.byref(h), C.byref(bw), C.byref(bh), C.byref(filt))
    if st != OK:
        raise PixlzrError(st, "malformed .pxlzr container")
    return dict(w=w.value, h=h.value, bw=bw.value, bh=bh.value, filter=filt.value)


def container_crop(data, c0: int, r0: int, nc: int, nr: int) -> bytes:
    """The .pxlzr file of the block window (c0, r0, nc, nr) of the file in `data` (any buffer: an mmap of a large file is
    read only in the header, the line table and the window's block rows), without decoding (pxz_container_crop)."""
    buf = np.frombuffer(data, np.uint8)
    n = lib().pxz_container_crop(ptr(buf), buf.size, c0, r0, nc, nr, None, 0)
    if n < 0:
        raise PixlzrError(int(n), "pxz_container_crop")
    out = np.empty(max(1, n), np.uint8)
    n = lib().pxz_container_crop(ptr(buf), buf.size, c0, r0, nc, nr, ptr(out), out.size)
    if n < 0:
        raise PixlzrError(int(n), "pxz_container_crop")
    return out[:n].tobytes()
