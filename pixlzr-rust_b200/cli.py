"""Command-line driver with the reference CLI's arguments and operation selection (src/bin/main.rs:7-265).

    python pixlzr_b200.py -i in.png -o out.pix -b 64 -k 1/2 -f lanczos3 --force

The operation follows from the two file extensions (main.rs:93-114): `.pix` / `.pixlzr` is the container, anything else an
image; an output without extension is a container.  As in the reference the blocks are only shrunk with `--force`
(main.rs:166-172, 204-210, 226-232, 256-262).  The pixel work runs on the GPU through the C ABI; image files are read and
written with Pillow on the host, the container with the library's host stage.
"""
from __future__ import annotations

import argparse
import os
import sys
from typing import List, Optional, Tuple

import numpy as np

from . import api

FILTERS = {"nearest": api.FilterType.Nearest, "triangle": api.FilterType.Triangle, "catmull-rom": api.FilterType.CatmullRom,
           "gaussian": api.FilterType.Gaussian, "lanczos3": api.FilterType.Lanczos3}


def build_parser() -> argparse.ArgumentParser:
    """clap definition of main.rs:7-43 (same flags, defaults and value names)."""
    p = argparse.ArgumentParser(prog="pixlzr", description="Pixlzr - A rust lib and CLI for the pixlzr image format")
    p.add_argument("-i", "--input", required=True, help="The input image file")
    p.add_argument("-o", "--output", required=True, help="The output image file")
    p.add_argument("-b", "--block-width", type=int, default=64, help="The width of each block")
    p.add_argument("--block-height", type=int, default=None, help="The height of each block")
    p.add_argument("-k", "--shrinking-factor", default="1",
                   help="The shrinking factor: [+|-][1/][D][.D]  If negative, is passed through max(0, 1 - x).")
    p.add_argument("-f", "--filter", choices=sorted(FILTERS), default="lanczos3",
                   help="The filter used when resizing the image blocks")
    p.add_argument("-d", "--direction-wise", type=lambda s: {"true": True, "false": False}[s.lower()], default=None,
                   metavar="true|false", help="Direction-wise scan")
    p.add_argument("--force", action="store_true", help="If image-2-image, force shrinking?")
    # extension (random access): not a flag of the reference
    p.add_argument("--region", type=parse_region, default=None, metavar="X,Y,W,H",
                   help="Decode only this pixel rectangle (.pix / .pixlzr -> image only)")
    # extension (rate control): not a flag of the reference
    p.add_argument("--payload-bytes", type=parse_payload_bytes, default=None, metavar="N",
                   help="Shrink with the largest factor whose block payload has at most N bytes, and print that factor "
                        "(image input, with --force; replaces -k)")
    # extension (rate control by error): not a flag of the reference
    p.add_argument("--target-psnr", type=parse_target_psnr, default=None, metavar="DB",
                   help="Shrink with the smallest factor whose decode (with -f) reaches DB dB PSNR against the input, and print "
                        "that factor, the payload bytes and the PSNR reached (image input, with --force; replaces -k)")
    # extension (optimised encode): not a flag of the reference
    p.add_argument("--optimal", action="store_true",
                   help="With --payload-bytes N or --target-psnr DB: choose every block's size on its own rather than one factor "
                        "for all (the least error within N bytes, or the fewest bytes reaching DB dB, decoded with -f), and print "
                        "the payload bytes and the PSNR reached (no -d: no metric is used)")
    # extension (decode error): not a flag of the reference
    p.add_argument("--psnr", action="store_true",
                   help="Decode what was written (with -f), compare it with the input image on the device and print the PSNR "
                        "and the largest difference (image input only)")
    return p


def parse_payload_bytes(s: str) -> int:
    try:
        n = int(s)
    except ValueError:
        raise argparse.ArgumentTypeError(f"expected a byte count, got {s!r}") from None
    if n < 0:
        raise argparse.ArgumentTypeError(f"expected a byte count >= 0, got {s!r}")
    return n


def parse_target_psnr(s: str) -> float:
    try:
        db = float(s)
    except ValueError:
        raise argparse.ArgumentTypeError(f"expected a PSNR in dB, got {s!r}") from None
    if db != db:
        raise argparse.ArgumentTypeError(f"expected a PSNR in dB, got {s!r}")
    return db


def parse_region(s: str) -> Tuple[int, int, int, int]:
    parts = s.split(",")
    try:
        x, y, w, h = (int(v) for v in parts)
    except ValueError:
        raise argparse.ArgumentTypeError(f"expected X,Y,W,H (four integers), got {s!r}") from None
    if x < 0 or y < 0 or w <= 0 or h <= 0:
        raise argparse.ArgumentTypeError(f"expected X, Y >= 0 and W, H > 0, got {s!r}")
    return x, y, w, h


def region_error(args) -> Optional[str]:
    """Why --region does not apply to this conversion, or None."""
    if args.region is not None and operation(args.input, args.output) != ("pix", "image"):
        return "--region decodes a rectangle of a .pix / .pixlzr file into an image: the input must be a container and the " \
               "output an image"
    return None


def payload_bytes_error(args) -> Optional[str]:
    """Why --payload-bytes does not apply to these arguments, or None."""
    if args.payload_bytes is None:
        return None
    if operation(args.input, args.output)[0] != "image":
        return "--payload-bytes chooses the factor of an encode: the input must be an image, not a container"
    if not args.force:
        return "--payload-bytes shrinks the blocks: it needs --force"
    if getattr(args, "factor_given", False):
        return "--payload-bytes chooses the shrinking factor: it cannot be combined with -k"
    if args.region is not None:
        return "--payload-bytes does not apply to a region decode"
    return None


def target_psnr_error(args) -> Optional[str]:
    """Why --target-psnr does not apply to these arguments, or None."""
    if getattr(args, "target_psnr", None) is None:
        return None
    if operation(args.input, args.output)[0] != "image":
        return "--target-psnr chooses the factor of an encode: the input must be an image, not a container"
    if not args.force:
        return "--target-psnr shrinks the blocks: it needs --force"
    if getattr(args, "factor_given", False):
        return "--target-psnr chooses the shrinking factor: it cannot be combined with -k"
    if args.payload_bytes is not None:
        return "--target-psnr and --payload-bytes each choose the factor: give one of them"
    if args.region is not None:
        return "--target-psnr does not apply to a region decode"
    return None


def optimal_error(args) -> Optional[str]:
    """Why --optimal does not apply to these arguments, or None."""
    if not getattr(args, "optimal", False):
        return None
    if args.payload_bytes is None and args.target_psnr is None:
        return "--optimal chooses every block's size for a budget: it needs --payload-bytes or --target-psnr"
    if args.direction_wise is not None:
        return "--optimal uses no metric: it cannot be combined with -d"
    return None


def psnr_error(args) -> Optional[str]:
    """Why --psnr does not apply to these arguments, or None."""
    if getattr(args, "psnr", False) and operation(args.input, args.output)[0] != "image":
        return "--psnr compares the decoded output with the input image: the input must be an image, not a container"
    return None


def parse_args(argv: Optional[List[str]] = None):
    """`-k -1/2`: the reference's clap option has allow_hyphen_values (main.rs:28-33); argparse needs `--opt=value`."""
    argv = list(sys.argv[1:] if argv is None else argv)
    out, i, factor_given = [], 0, False
    while i < len(argv):
        if argv[i] in ("-k", "--shrinking-factor") and i + 1 < len(argv):
            out.append("--shrinking-factor=" + argv[i + 1])
            factor_given = True
            i += 2
        else:
            factor_given = factor_given or argv[i].startswith("--shrinking-factor=")
            out.append(argv[i])
            i += 1
    args = build_parser().parse_args(out)
    args.factor_given = factor_given  # --payload-bytes refuses an explicit -k, even `-k 1`
    return args


def kind_of(path: str, default: str) -> str:
    """main.rs:93-114: "pix" for .pix / .pixlzr (any case), "image" for another extension, `default` without one."""
    ext = os.path.splitext(path)[1]
    if not ext:
        return default
    return "pix" if ext[1:].lower() in ("pix", "pixlzr") else "image"


def operation(input_path: str, output_path: str) -> Tuple[str, str]:
    return kind_of(input_path, "image"), kind_of(output_path, "pix")


def _open_image(path: str) -> np.ndarray:
    from PIL import Image
    im = Image.open(path)
    if im.mode not in ("RGB", "RGBA"):
        im = im.convert("RGBA" if "A" in im.getbands() or "transparency" in im.info else "RGB")
    return np.ascontiguousarray(np.array(im))


def _save_image(path: str, pixels: np.ndarray) -> None:
    from PIL import Image
    Image.fromarray(pixels).save(path)


def _maybe_shrink(pix: api.Pixlzr, args, shrink_by: float) -> None:
    if not args.force:
        return
    if args.direction_wise:
        pix.shrink_directionally(FILTERS[args.filter], shrink_by)
    else:
        pix.shrink_by(FILTERS[args.filter], shrink_by)


def run(args) -> None:
    bw = args.block_width
    bh = args.block_height if args.block_height is not None else bw
    filt = FILTERS[args.filter]
    shrink_by = api.parse_shrinking_factor(args.shrinking_factor)
    src, dst = operation(args.input, args.output)
    err = region_error(args) or payload_bytes_error(args) or target_psnr_error(args) or optimal_error(args) or psnr_error(args)
    if err:
        raise ValueError(err)
    if args.optimal or args.target_psnr is not None:
        _run_budgeted(args, bw, bh, filt, dst)
        return
    if args.payload_bytes is not None:
        _run_sized(args, bw, bh, filt, src, dst)
        return
    if args.region is not None and not (args.force and args.direction_wise):
        with open(args.input, "rb") as f:
            _save_image(args.output, api.Pixlzr.decode_vec_region_to_image(f.read(), filt, *args.region))
        return
    # the two plain conversions run with the container stage on the device (same bytes / pixels as the general path)
    if src == "image" and dst == "pix" and args.force:
        with open(args.output, "wb") as f:
            f.write(api.Pixlzr.encode_image_to_vec(_open_image(args.input), bw, bh, filt, shrink_by, bool(args.direction_wise)))
        return
    # pix -> image: shrink_by leaves a decoded file alone (every block carries a value, pixlzr.rs:168-170), so --force only
    # matters with -d true: shrink_directionally has no such check (pixlzr.rs:187-205) and re-shrinks the decoded blocks —
    # that case takes the general path below
    if src == "pix" and dst == "image" and not (args.force and args.direction_wise):
        with open(args.input, "rb") as f:
            _save_image(args.output, api.Pixlzr.decode_vec_to_image(f.read(), filt))
        return
    if src == "image":                                   # image_to_pix / image_to_image (main.rs:142-214)
        pix = api.Pixlzr.from_image(_open_image(args.input), bw, bh)
    elif dst == "image":                                 # pix_to_image (main.rs:216-240)
        pix = api.Pixlzr.open(args.input)
    else:                                                # pix_to_pix re-tiles the decoded image (main.rs:242-265)
        pix = api.Pixlzr.from_image(api.Pixlzr.open(args.input).to_image(filt), bw, bh)
    _maybe_shrink(pix, args, shrink_by)
    if dst == "pix":
        pix.save(args.output)
    elif args.region is not None:
        _save_image(args.output, pix.to_image_region(filt, *args.region))
    else:
        _save_image(args.output, pix.to_image(filt))


def _run_sized(args, bw: int, bh: int, filt, src: str, dst: str) -> None:
    """image -> container / image with the factor chosen for --payload-bytes; prints the factor in a form -k reads back."""
    image = _open_image(args.input)
    if dst == "pix":
        data, k = api.Pixlzr.encode_image_to_vec_sized(image, bw, bh, filt, args.payload_bytes, bool(args.direction_wise))
        with open(args.output, "wb") as f:
            f.write(data)
    else:
        pix = api.Pixlzr.from_image(image, bw, bh)
        k = pix.shrink_to_size(filt, args.payload_bytes, bool(args.direction_wise))
        _save_image(args.output, pix.to_image(filt))
    print(f"shrinking factor: {api.format_shrinking_factor(k)}")


def _run_budgeted(args, bw: int, bh: int, filt, dst: str) -> None:
    """image -> container / image for a budget on the decode with -f (the filter a decoder of the written file uses).  Without
    --optimal: the smallest factor whose decode reaches --target-psnr; prints the factor in a form -k reads back.  With
    --optimal: every block's size chosen for --payload-bytes (the least error within N bytes) or --target-psnr (the fewest
    bytes reaching it).  Then prints the payload bytes and the PSNR reached."""
    image = _open_image(args.input)
    ctx = api.default_context()
    img = ctx.image_upload(image)
    k = nbytes = None
    try:
        samples = img.w * img.h * img.c
        if not args.optimal:
            metric = api.N.METRIC_SOBEL_DIR if args.direction_wise else api.N.METRIC_OKLAB_MAD
            pl, k, sse = img.shrink_to_error(bw, bh, metric, api.sse_budget(args.target_psnr, samples), int(filt), int(filt), 0)
        elif args.payload_bytes is not None:
            pl, nbytes, sse = img.rdo_shrink_to_size(bw, bh, args.payload_bytes, int(filt), int(filt))
        else:
            pl, nbytes, sse = img.rdo_shrink_to_error(bw, bh, api.sse_budget(args.target_psnr, samples), int(filt), int(filt))
    finally:
        img.free()
    try:
        if nbytes is None:
            nbytes = pl.info()["bytes"]
        if dst == "pix":
            with open(args.output, "wb") as f:
                f.write(pl.to_container(0, True))
        else:
            _save_image(args.output, pl.expand(int(filt)))
    finally:
        pl.free()
    if k is not None:
        print(f"shrinking factor: {api.format_shrinking_factor(k)}")
    print(f"payload bytes: {nbytes}")
    print(f"psnr: {format_psnr(api.psnr_of(sse, samples))} dB")


def format_psnr(psnr: float) -> str:
    return "inf" if psnr == float("inf") else f"{psnr:.6f}"


def report_psnr(args) -> None:
    """Decodes the written output with -f and prints its error against the input image (computed on the device)."""
    bw = args.block_width
    bh = args.block_height if args.block_height is not None else bw
    source = _open_image(args.input)
    if operation(args.input, args.output)[1] == "pix":
        ctx = api.default_context()
        with open(args.output, "rb") as f:
            pl, _ = ctx.payload_from_container(f.read())
        try:
            rep = api.payload_error(pl, source, FILTERS[args.filter])
        finally:
            pl.free()
    else:
        rep = api.image_error(_open_image(args.output), source, bw, bh)
    print(f"psnr: {format_psnr(rep.psnr)} dB, max error: {rep.max_error}")


def main(argv: Optional[List[str]] = None) -> int:
    args = parse_args(argv)
    err = region_error(args) or payload_bytes_error(args) or target_psnr_error(args) or optimal_error(args) or psnr_error(args)
    if err:
        print(f"pixlzr: {err}", file=sys.stderr)
        return 2
    try:
        run(args)
        if args.psnr:
            report_psnr(args)
    except FileNotFoundError as e:
        print(f"Could not open the image [ {e.filename} ]", file=sys.stderr)
        return 1
    return 0
