"""IsMatch / GetDecompressedSize parity on the GPU library (magic checks on the host side of the library, the
LZ10 / LZ11 / PRS token-walk heuristics on the device), and the reference's DataRecognitionTest through the
interface mirror (CompressionAlgorithmTest.cs:60-80)."""
import io

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests.util import MATCHABLE, SIZED_FORMATS, decoded_size_blobs, fmt_id, is_match_blobs, rom_like_image, synth

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("fmt", MATCHABLE, ids=fmt_id)
def test_is_match_parity(codec, oracle, bmp, fmt):
    blobs = is_match_blobs(oracle, bmp, fmt)
    got = codec.is_match_batch(fmt, blobs)
    ref = np.array([oracle.is_match(fmt, b) for b in blobs])
    bad = np.nonzero(got != ref)[0]
    assert len(bad) == 0, f"{fmt_id(fmt)}: {len(bad)} of {len(blobs)} differ, first #{bad[0]} gpu={got[bad[0]]} ref={ref[bad[0]]} blob={blobs[bad[0]][:24].hex()} len={len(blobs[bad[0]])}"
    assert got.sum() > 0


@pytest.mark.parametrize("fmt", SIZED_FORMATS, ids=fmt_id)
def test_decoded_size_parity(codec, oracle, fmt):
    blobs = decoded_size_blobs(oracle, fmt)
    for opts in (None, A.make_opts(byte_order=A.ENDIAN_LITTLE), A.make_opts(byte_order=A.ENDIAN_BIG)):
        size, status = codec.decoded_size_batch(fmt, blobs, opts)
        for b, s, st in zip(blobs, size, status):
            rs, rst = oracle.decoded_size(fmt, b, opts)
            assert (int(s), int(st)) == (rs, rst) or (st != 0 and rst != 0), (fmt_id(fmt), b[:16].hex(), int(s), int(st), rs, rst)


def test_data_recognition_through_the_mirror(codec, oracle):
    """256 zero bytes at CompressionSettings.Fastest: Compress on the GPU, IsMatch true, GetDecompressedSize 0x100,
    Decompress round trip — the reference's DataRecognitionTest + EncodingAndDecodingMatchTest shape."""
    from auroralib.compression_b200 import BLZ, LZ10, LZ11, LZ40, LZ60, LZSS, MIO0, SMSR00, CompressionSettings, LZHudson, Yay0, Yaz0, Yaz1
    from tests.util import end_position
    data = bytes(0x100)
    for cls in (Yaz0, Yaz1, Yay0, MIO0, LZ10, LZ11, LZSS, LZHudson, LZ40, LZ60, SMSR00, BLZ):
        algo = cls()
        comp = algo.Compress(data, None, CompressionSettings.Fastest)
        ref, st = oracle.encode(algo.FORMAT, data, A.make_opts(quality=0))
        assert comp.getvalue() == ref, cls.__name__
        assert algo.IsMatch(comp)
        assert algo.GetDecompressedSize(comp) == 0x100
        assert comp.tell() == 0
        out = algo.Decompress(comp)
        assert out.getvalue() == data and comp.tell() == end_position(algo.FORMAT, ref)


def test_mirror_streams_and_exceptions(codec, oracle, bmp):
    from auroralib.compression_b200 import (LZ4, LZ10, LZO, PRS, DecompressedSizeException, EndOfStreamException,
                                            InvalidIdentifierException, Snappy, Yaz0)
    raw = bmp[:30000]
    # source consumed from its current position and left just past the compressed bytes; destination appended
    comp, _ = oracle.encode(A.FMT_YAZ0, raw, A.make_opts(quality=8))
    src = io.BytesIO(b"junk" + comp + b"tail")
    src.seek(4)
    dst = io.BytesIO(b"head")
    dst.seek(4)
    Yaz0().Decompress(src, dst)
    assert dst.getvalue() == b"head" + raw and src.tell() == 4 + len(comp)
    for cls, fmt in ((LZ4, A.FMT_LZ4), (LZO, A.FMT_LZO), (Snappy, A.FMT_SNAPPY), (PRS, A.FMT_PRS)):   # no size header: device size pre-pass
        c, _ = oracle.encode(fmt, raw, A.make_opts(quality=4))
        assert cls().Decompress(io.BytesIO(c)).getvalue() == raw
    with pytest.raises(InvalidIdentifierException):
        LZ10().Decompress(io.BytesIO(b"\x11" + comp))
    lz, _ = oracle.encode(A.FMT_LZ10, raw, A.make_opts(quality=8))
    with pytest.raises(EndOfStreamException):
        LZ10().Decompress(io.BytesIO(lz[:1000]))
    bad = bytearray(lz)
    bad[1:4] = (29990).to_bytes(3, "little")
    try:
        LZ10().Decompress(io.BytesIO(bytes(bad)))
    except DecompressedSizeException as e:
        assert e.expected == 29990
    le = Yaz0()
    le.FormatByteOrder = 0
    c = le.Compress(raw)
    assert c.getvalue()[4:8] == len(raw).to_bytes(4, "little")
    assert Yaz0().Decompress(c).getvalue() == raw   # default Big: the swapped-size retry (Yaz0.cs:67-78)


def test_offset_scan_of_a_rom_like_image(codec, oracle, bmp):
    """The CLI's `-scan` (ScanDecompressCommand.cs:23-39) as one pass: IsMatch at every offset of an image that holds a few
    compressed assets between junk, then decode at the hits and resume after the consumed bytes."""
    rng = np.random.default_rng(77)
    assets = [bmp[1000:9000], bytes(3000), synth(rng, 5000, 0), synth(rng, 2500, 2)]
    for fmt in (A.FMT_YAZ0, A.FMT_LZ10, A.FMT_LZ11, A.FMT_MIO0, A.FMT_LZ4, A.FMT_PRS):
        image, starts = rom_like_image(oracle, rng, fmt, assets)
        got = codec.scan_offsets(fmt, image)
        ref = np.array([oracle.is_match(fmt, image[i:]) for i in range(len(image))])
        assert (got == ref).all(), (fmt_id(fmt), int((got != ref).sum()))
        if fmt in (A.FMT_YAZ0, A.FMT_MIO0, A.FMT_LZ4):   # magic formats hit every asset (the token-walk heuristics may not, like the reference)
            assert all(got[s] for s in starts), fmt_id(fmt)
        if fmt in (A.FMT_YAZ0, A.FMT_MIO0):   # magic formats: walk the bitmap like the CLI does
            found, i = [], 0
            while i < len(image):
                if got[i]:
                    outs, out_len, consumed, status = codec.decode_batch(fmt, [image[i:]], [1 << 16])
                    if status[0] == 0:
                        found.append(outs[0])
                        i += int(consumed[0])
                        continue
                i += 1
            assert found == assets
