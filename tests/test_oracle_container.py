"""Pins the oracle's container layer (SURVEY section 8f row N2: signature, chunk framing, per-chunk
CRC-32, IHDR / PLTE / tRNS parsing, IDAT concatenation and framing) against the reference's vectors:
its 14 malformed inputs with the errors ErrorHandling.swift expects, every PngSuite / CgBI golden
through the file-level entry point, and its committed level-9 outputs byte for byte as whole files."""
import hashlib
import json
import os
import struct
import zlib

import pytest

import container_cases as cc
import pngio
from conftest import GOLDEN

PNGSUITE = sorted(f for f in os.listdir(os.path.join(GOLDEN, "pngsuite")) if f.endswith(".png"))
IOS = sorted(f for f in os.listdir(os.path.join(GOLDEN, "ios")) if f.endswith(".png"))
DIGESTS = json.load(open(os.path.join(GOLDEN, "pngsuite_rgba.json")))
IOS_DIGESTS = json.load(open(os.path.join(GOLDEN, "ios_rgba.json")))
ENC = json.load(open(os.path.join(GOLDEN, "encode.json")))
KEPT = sorted(f[4:] for f in os.listdir(os.path.join(GOLDEN, "encode")) if f.startswith("out-"))
SAMPLED = sorted(os.listdir(os.path.join(GOLDEN, "outputs")))


def invalid_cases(o):
    """(file, status, a, b) from Sources/PNGIntegrationTests/ErrorHandling.swift:7-76"""
    sig = [(n, (o.ERR_LEX_INVALID_SIGNATURE,)) for n in
           ("xs1n0g01", "xs2n0g01", "xs4n0g01", "xs7n0g01", "xcrn0g04", "xlfn0g04")]
    return sig + [
        ("xhdn0g08", (o.ERR_LEX_INVALID_CHUNK_CHECKSUM, 1129534797, 1443964200)),
        ("xcsn0g01", (o.ERR_LEX_INVALID_CHUNK_CHECKSUM, 1129534797, 3492746441)),
        ("xc1n0g08", (o.ERR_PARSE_HEADER_PIXEL_FORMAT_CODE, 8, 1)),
        ("xc9n2c08", (o.ERR_PARSE_HEADER_PIXEL_FORMAT_CODE, 8, 9)),
        ("xd0n2c08", (o.ERR_PARSE_HEADER_PIXEL_FORMAT_CODE, 0, 2)),
        ("xd3n2c08", (o.ERR_PARSE_HEADER_PIXEL_FORMAT_CODE, 3, 2)),
        ("xd9n2c08", (o.ERR_PARSE_HEADER_PIXEL_FORMAT_CODE, 99, 2)),
        ("xdtn0g01", (o.ERR_DECODE_REQUIRED_CHUNK, o.fourcc("IDAT"), o.fourcc("IEND"))),
    ]


def test_reference_error_cases(orc):
    cases = invalid_cases(orc)
    assert sorted(n + ".png" for n, _ in cases) == sorted(os.listdir(os.path.join(GOLDEN, "invalid")))
    for name, want in cases:
        data = open(os.path.join(GOLDEN, "invalid", name + ".png"), "rb").read()
        for info in (orc.png_inspect(data), orc.png_decompress(data)[0]):
            got = (info.status, info.a, info.b)
            assert got[: len(want)] == want, (name, got)


@pytest.mark.parametrize("sub,names,digests", [("pngsuite", PNGSUITE, DIGESTS), ("ios", IOS, IOS_DIGESTS)])
def test_goldens_through_decompress(orc, sub, names, digests):
    """PNG.Image.decompress(path:) + unpack(as: RGBA<UInt16>) == golden, from the file bytes"""
    for name in names:
        data = open(os.path.join(GOLDEN, sub, name), "rb").read()
        info, storage = orc.png_decompress(data)
        assert info.status == 0, (name, info.status)
        st, px = orc.unpack(storage, orc.make_format(**info.fields()), orc.TARGET_RGBA16)
        assert st == 0 and hashlib.sha256(px).hexdigest() == digests[name]["sha256"], name
        # the header / format the test-side parser derives agree with the oracle's
        png = pngio.parse(data)
        assert (info.width, info.height, info.depth, info.color, bool(info.interlaced), bool(info.standard)) == \
               (png.width, png.height, png.depth, png.color, png.interlaced, png.cgbi)
        assert info.idat_bytes == len(png.idat) and info.fields() == pngio.format_fields(png)


@pytest.mark.parametrize("name", KEPT)
def test_level9_outputs_whole_file(orc, name):
    """Tests/Outputs/<name> == image.compress(level: 9) of Tests/Baselines/<name>, every byte of the
    file: signature, IHDR, PLTE, IDAT chunks of 65544 bytes with their CRCs, IEND"""
    base = open(os.path.join(GOLDEN, "encode", "in-" + name), "rb").read()
    want = open(os.path.join(GOLDEN, "encode", "out-" + name), "rb").read()
    info, storage = orc.png_decompress(base)
    assert info.status == 0
    got = orc.png_compress(storage, info.width, info.height, orc.make_format(**info.fields()), bool(info.interlaced), 9)
    assert hashlib.sha256(got).hexdigest() == ENC[name]["file_sha256"]
    assert got == want


def test_level9_sampled_outputs_whole_file(orc):
    """every Tests/Outputs file kept under golden/ (encode.json holds the digests of all 28) is
    image.compress(level: 9) of its image, whole.  Where the Tests/Baselines input is not kept
    (outputs/*), the image is decompressed from the output: the encoder is lossless."""
    cases = [(n, os.path.join(GOLDEN, "encode", "in-" + n)) for n in KEPT] + \
            [(n, os.path.join(GOLDEN, "outputs", n)) for n in SAMPLED]
    assert len(cases) == 6 and len(ENC) == 28
    for name, src in cases:
        base = open(src, "rb").read()
        info, storage = orc.png_decompress(base)
        assert info.status == 0, name
        got = orc.png_compress(storage, info.width, info.height, orc.make_format(**info.fields()), bool(info.interlaced), 9)
        assert len(got) == ENC[name]["file_bytes"] and hashlib.sha256(got).hexdigest() == ENC[name]["file_sha256"], name


def test_lexing_and_ordering_rules(orc):
    o = orc
    _chunk, _png = cc.chunk, cc.png
    ihdr, plte, idat, iend = cc.IHDR, cc.PLTE, cc.IDAT, cc.IEND
    ok = _png([ihdr, plte, _chunk(b"tRNS", b"\x80"), idat, iend])
    info, storage = o.png_decompress(ok)
    assert info.status == 0 and storage == bytes([0, 1, 1, 0])
    assert info.fields()["palette"] == bytes([0, 1, 2, 0x80, 3, 4, 5, 255])
    cases = cc.structural_cases(o)
    for data, want in cases:
        for info in (o.png_inspect(data), o.png_decompress(data)[0]):
            got = (info.status, info.a, info.b)
            assert got[: len(want)] == want, (data[:40], got, want)
    # decoder errors keep their place in stream order: bad deflate data in the first IDAT wins over a
    # CRC error in a later chunk; a CRC error in the IDAT itself wins over its contents
    _chunk, _png = cc.chunk, cc.png
    ihdr, plte, iend = cc.IHDR, cc.PLTE, cc.IEND
    bad = cc.chunk(b"IDAT", b"\x78\x9c\x07")
    later = cc.chunk(b"tEXt", b"k\0v", crc=1)
    info, _ = o.png_decompress(_png([ihdr, plte, bad, later, iend]))
    assert info.status == o.ERR_BLOCK_TYPE
    assert o.png_inspect(_png([ihdr, plte, bad, later, iend])).status == o.ERR_LEX_INVALID_CHUNK_CHECKSUM
    info, _ = o.png_decompress(_png([ihdr, plte, _chunk(b"IDAT", b"\x78\x9c\x07", crc=5), iend]))
    assert info.status == o.ERR_LEX_INVALID_CHUNK_CHECKSUM and info.a == 5
    # truncated image data: IEND arrives while the decoder still wants input
    short = _chunk(b"IDAT", zlib.compress(bytes([0, 0, 1, 0, 1, 0]))[:-6])
    info, _ = o.png_decompress(_png([ihdr, plte, short, iend]))
    assert info.status == o.ERR_PNG_INCOMPLETE_DATASTREAM


def test_compress_writes_cgbi_and_transparency(orc):
    """[CgBI] IHDR [PLTE] [tRNS] IDAT.. IEND; the file decompresses to the same storage and format"""
    import numpy as np
    rng = np.random.default_rng(3)
    for fields, w, h in ((dict(color=6, depth=8, bgr=True), 5, 4), (dict(color=2, depth=8, bgr=True, key=(3, 2, 1)), 4, 4),
                         (dict(color=0, depth=4, key=(9,)), 7, 3), (dict(color=2, depth=16, key=(1, 2, 3)), 3, 3),
                         (dict(color=3, depth=2, palette=bytes([1, 2, 3, 255, 4, 5, 6, 7, 8, 9, 10, 255])), 9, 2)):
        fmt = orc.make_format(**fields)
        ch = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}[fields["color"]]
        n = w * h * ch * (2 if fields["depth"] == 16 else 1)
        top = 3 if fields["color"] == 3 else (1 << min(fields["depth"], 8))
        storage = rng.integers(0, top, n, dtype=np.uint8).tobytes()
        for interlaced in (False, True):
            data = orc.png_compress(storage, w, h, fmt, interlaced, 6, idat_chunk=16)
            info, back = orc.png_decompress(data)
            assert info.status == 0 and back == storage and bool(info.interlaced) == interlaced
            want = dict(bgr=False, key=None, palette=None)
            want.update(fields)
            assert info.fields() == want
            png = pngio.parse(data)  # independent chunk walk: CRCs, chunk order, IDAT framing
            assert png.chunks[0] == (b"CgBI" if fields.get("bgr") else b"IHDR") and png.chunks[-1] == b"IEND"
            assert max(len(c) for c in [png.idat]) > 0 and png.chunks.count(b"IDAT") == (len(png.idat) + 15) // 16
