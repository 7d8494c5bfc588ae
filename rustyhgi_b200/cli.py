"""`hgi` command line with the reference's sub-commands and flags (src/options.rs:13-64, src/main.rs:41-134):

    hgi encode -i <image> -o <archive.hgi> [-l 4] [-q medium]
    hgi decode -i <archive.hgi> -o <image> [--scale K] [--region X,Y,W,H]
    hgi test <image> [-s suffix] [-l 4] [-q medium]

Always Crossed + Linear like the reference (src/main.rs:43-45,67,76-78).  File decoding/encoding is PIL
on the host; RGB->luma, the codec and the error metrics run on the GPU through libhgi_b200.so; the
archive container is hgi_archive_* (host).  Errors are printed and the exit code stays 0, exactly like
`main` (src/main.rs:130-134).
"""
import argparse
import io
import os
import sys

import numpy as np

from . import api


def _open_luma(path):
    """`image::open(path)?.to_luma()` (src/main.rs:42,74)."""
    from PIL import Image
    im = Image.open(path)
    if im.mode == "L":
        return np.array(im)
    return api.rgb_to_luma(np.array(im.convert("RGB")))


def _level(text):
    try:
        return api.QuantizationLevel.parse(text)       # clap arg_enum!: case-insensitive variant names
    except ValueError as e:
        raise argparse.ArgumentTypeError(str(e))


def _encoding_options(p):
    p.add_argument("-l", "--level", type=int, default=4)                      # src/options.rs:55-56
    p.add_argument("-q", "--quantizator", type=_level, default="medium")      # src/options.rs:58-64
    # not in the reference: which DEFLATE encoder writes the payload.  "rle" = GPU-built token tables + host bit
    # packing (zlib-9 size on residual planes, ~100x faster); "deflate" = zlib level 9, the closest stand-in for
    # flate2's Compression::best().  Every choice is a raw DEFLATE stream the reference reads.
    p.add_argument("--entropy", choices=("rle", "deflate", "huffman"), default="rle")


def _scale(text):
    k = int(text)
    if not 0 <= k <= 31:
        raise argparse.ArgumentTypeError("scale must be 0..31")
    return k


def _region(text):
    try:
        v = tuple(int(t) for t in text.split(","))
    except ValueError:
        v = ()
    if len(v) != 4 or min(v) < 0:
        raise argparse.ArgumentTypeError("region must be X,Y,W,H (non-negative integers)")
    return v


def build_parser():
    ap = argparse.ArgumentParser(prog="hgi", description="Hierarchical Grid Interpolation codec (B200)")
    sub = ap.add_subparsers(dest="cmd", required=True)
    enc = sub.add_parser("encode")
    enc.add_argument("-i", "--input", required=True)
    enc.add_argument("-o", "--output", required=True)
    _encoding_options(enc)
    dec = sub.add_parser("decode")
    dec.add_argument("-i", "--input", required=True)
    dec.add_argument("-o", "--output", required=True)
    # not in the reference: scalable decode.  The archive's DEFLATE payload is in raster order, so it is still
    # inflated whole on the host; only the GPU decode is limited to the rows and columns the output depends on.
    dec.add_argument("--scale", type=_scale, default=0,
                     help="write the image at 1/2^K resolution (every 2^K-th pixel of every 2^K-th row); the "
                          "archive is still inflated whole")
    dec.add_argument("--region", type=_region, default=None, metavar="X,Y,W,H",
                     help="write only this rectangle, in the coordinates of the (scaled) image")
    tst = sub.add_parser("test")
    tst.add_argument("input")
    tst.add_argument("-s", "--suffix", default="")                              # src/options.rs:34-35
    _encoding_options(tst)
    return ap


def encode(a):                                            # src/main.rs:41-61
    image = _open_luma(a.input)
    h, w = image.shape
    grid = api.Encoder(api.Crossed, api.Linear(a.quantizator), a.level).encode(image)
    md = api.Metadata(a.quantizator, api.InterpolationType.Crossed, w, h, a.level)
    with open(a.output, "wb") as f:
        api.Archive(md, grid).serialize_to_writer(f, entropy=a.entropy)


def decode(a):                                            # src/main.rs:63-71
    from PIL import Image
    with open(a.input, "rb") as f:
        arch = api.Archive.deserialize_from_reader(f)
    m = arch.metadata
    if a.scale or a.region is not None:
        image = api.Decoder(api.Crossed).decode_region((m.width, m.height), m.scale_level, arch.grid, a.region, a.scale)
    else:
        image = api.Decoder(api.Crossed).decode((m.width, m.height), m.scale_level, arch.grid)
    Image.fromarray(image, "L").save(a.output)


def test(a, out=None):                                    # src/main.rs:73-120
    out = out or sys.stdout
    from PIL import Image
    before = _open_luma(a.input)
    h, w = before.shape
    grid = api.Encoder(api.Crossed, api.Linear(a.quantizator), a.level).encode(before)
    after = api.Decoder(api.Crossed).decode((w, h), a.level, grid)
    m = api.error_metrics(before, after)
    buf = io.BytesIO()
    api.Archive(api.Metadata(a.quantizator, api.InterpolationType.Crossed, w, h, a.level), grid).serialize_to_writer(buf, entropy=a.entropy)
    uncompressed, compressed = w * h, len(buf.getvalue())
    print(f"Uncompressed: {uncompressed // 1024} kb", file=out)               # src/main.rs:108-111
    print(f"Compressed:   {compressed // 1024} kb", file=out)
    print(f"Ratio:        {uncompressed / compressed:.2f}", file=out)
    print(f"SD:           {m['sd']:.2f}", file=out)
    stem = os.path.splitext(os.path.basename(a.input))[0] + a.suffix          # src/main.rs:113
    Image.fromarray(after, "L").save(stem + ".png")
    with open(stem + ".hgi", "wb") as f:
        f.write(buf.getvalue())


def main(argv=None):
    a = build_parser().parse_args(argv)
    try:
        {"encode": encode, "decode": decode, "test": test}[a.cmd](a)
    except Exception as e:                                 # src/main.rs:130-134: print, exit code 0
        print(f"An error occured: {e}", file=sys.stderr)


if __name__ == "__main__":
    main()
