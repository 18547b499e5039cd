"""CPU tests: the oracle against every golden vector / known answer the reference holds for the hot path
(SURVEY.md §8c, BASELINE.md §2).  These pin the checker before the GPU parity tests trust it."""
import hashlib
import os

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests.util import ALL_FORMATS, SIZED_FORMATS, end_position, fmt_id, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_fixture_integrity(bmp, test_lz):
    assert len(bmp) == 1048726 and len(test_lz) == 285929
    assert hashlib.sha256(bmp).hexdigest() == "5c8809e6059937c47544839bfa9f8d70a878574a0442c903e8353b2456757ccd"


def test_hash_known_answers(oracle):
    # published test vectors of XXH32 / XXH64 (seed 0) and CRC-32C
    assert oracle.xxh32(b"") == 0x02CC5D05 and oracle.xxh64(b"") == 0xEF46DB3751D8E999
    assert oracle.xxh32(b"a") == 0x550D7456 and oracle.xxh64(b"a") == 0xD24EC4F1A98C6E5B
    assert oracle.crc32c(b"123456789") == 0xE3069283


def test_lzss_static_decoding(oracle, bmp, test_lz):
    """LzssStaticDecodingTest (CompressionTest/CompressionAlgorithmTest.cs:30-48): the only known-answer decode."""
    opts = A.make_opts(lzss=A.lz_props_bits(10, 6, 2))
    size, st = oracle.decoded_size(A.FMT_LZSS, test_lz, opts)
    assert st == 0 and size == 1048726
    out, out_len, consumed, status = oracle.decode(A.FMT_LZSS, test_lz, size, opts)
    assert status == 0 and consumed == len(test_lz)
    assert oracle.xxh64(out) == 11520079745250749767
    assert out == bmp


Q0_SIZES = {A.FMT_YAZ0: 183160, A.FMT_YAY0: 183160, A.FMT_LZ10: 261953, A.FMT_MIO0: 261898, A.FMT_LZSS: 261898,
            A.FMT_LZ11: 179455, A.FMT_LZ4_LEGACY: 175023, A.FMT_LZO: 161204, A.FMT_SNAPPY: 209184, A.FMT_PRS: 165729,
            A.FMT_LZ40: 179488, A.FMT_LZ60: 179488, A.FMT_LZ00: 261946, A.FMT_BLZ: 345456}


@pytest.mark.parametrize("fmt", sorted(Q0_SIZES), ids=fmt_id)
def test_published_q0_ratios(oracle, bmp, fmt):
    """Benchmarks.md Q0 ratios on the first 1 024 000 bytes of Test.bmp, to the byte (BASELINE.md §2)."""
    raw = bmp[:1024000]
    comp, st = oracle.encode(fmt, raw, A.make_opts(quality=0))
    assert st == 0 and len(comp) == Q0_SIZES[fmt]
    published = {A.FMT_YAZ0: 17.89, A.FMT_YAY0: 17.89, A.FMT_LZ10: 25.58, A.FMT_MIO0: 25.58, A.FMT_LZSS: 25.58, A.FMT_LZ11: 17.52,
                 A.FMT_LZ4_LEGACY: 17.09, A.FMT_LZO: 15.74, A.FMT_SNAPPY: 20.43, A.FMT_PRS: 16.18,
                 A.FMT_LZ40: 17.53, A.FMT_LZ60: 17.53, A.FMT_LZ00: 25.58, A.FMT_BLZ: 33.74}[fmt]   # (LZ60 is LZ40 under another identifier)
    assert round(100 * len(comp) / len(raw), 2) == published
    out, out_len, consumed, status = oracle.decode(fmt, comp, len(raw))
    assert status == 0 and out == raw and consumed == end_position(fmt, comp)


def test_q15_and_whole_file_sizes(oracle, bmp):
    """LZO Q15 equals the published 11.29 %; whole-file Yaz0 / LZ10 sizes of the survey-time restatement."""
    comp, st = oracle.encode(A.FMT_LZO, bmp[:1024000], A.make_opts(quality=15))
    assert len(comp) == 115629
    for fmt, exp in ((A.FMT_YAZ0, {0: 183638, 8: 175231, 15: 153194}), (A.FMT_LZ10, {0: 265004, 8: 251850, 15: 235988})):
        for q, e in exp.items():
            comp, st = oracle.encode(fmt, bmp, A.make_opts(quality=q))
            assert st == 0 and len(comp) == e


def test_q15_ratios_within_a_tenth_of_a_point_of_the_published_ones(oracle, bmp):
    """Benchmarks.md Q15 ratios on the first 1 024 000 bytes of Test.bmp.  LZO is exact (test above); the 4 KiB-window formats
    come out 0.07-0.08 percentage points SMALLER than published (LZ10 22.76 vs 22.84 %, LZ11 14.20 vs 14.28 %, Yaz0 14.93 vs
    15.01 %) — consistently, so either Benchmarks.md predates the mounted sources or the chain walk differs in a corner that
    only deep chains reach ("parity unpinned" beyond this tolerance, DESIGN.md section 2).  The Q0 ratios are exact.
    Round 2 chased the drift: the restatement was diffed by hand against LzChainMatchFinder.cs:42-357 again (no difference),
    and a scan of the finder parameters through the oracle's investigation knobs (ORACLE_LAZY 3..18, ORACLE_MAXCHAIN 64..2048,
    ORACLE_HASHBITS 16..20, ORACLE_NO_MINTABLE) never lands on the published sizes.  The gap is a near-constant 791-818 BYTES
    for LZ10 / LZ11 / Yaz0 alike (233 068 vs 233 882, 145 409 vs 146 227, 152 911 vs 153 702) although their token formats
    differ — about 800 fewer 3-byte matches, i.e. the small-match (min table) path of the finder that produced Benchmarks.md
    behaved differently from the mounted sources (no git history is mounted to date it).  LZO's Q15 size, which never uses
    that path (MinLength 3 matches come from the 4-byte chains there too, but its window is 48 KiB with a 64 Ki chain ring),
    is exact."""
    published = {A.FMT_LZ10: 22.84, A.FMT_LZ11: 14.28, A.FMT_YAZ0: 15.01, A.FMT_YAY0: 15.01, A.FMT_MIO0: 22.84, A.FMT_LZSS: 22.84,
                 A.FMT_LZ40: 14.28, A.FMT_LZ00: 22.84, A.FMT_BLZ: 22.86, A.FMT_PRS: 13.83}
    raw = bmp[:1024000]
    for fmt, pct in published.items():
        comp, st = oracle.encode(fmt, raw, A.make_opts(quality=15))
        assert st == 0 and abs(100 * len(comp) / len(raw) - pct) <= 0.10, (fmt_id(fmt), 100 * len(comp) / len(raw), pct)


@pytest.mark.parametrize("fmt", ALL_FORMATS, ids=fmt_id)
def test_reference_round_trips(oracle, bmp, fmt):
    """EncodingAndDecodingMatchTest_{10b, 10kb_Balanced, 10kb_Maximum, 1MB_Fastest} (:81-130)."""
    for n, q in ((10, 4), (10240, 8), (10240, 15), (1048576, 0)):
        comp, st = oracle.encode(fmt, bmp[:n], A.make_opts(quality=q))
        assert st == 0
        out, out_len, consumed, status = oracle.decode(fmt, comp, n)
        assert status == 0 and out == bmp[:n] and consumed == end_position(fmt, comp)


def test_lz4_frame_whole_file(oracle, bmp):
    """EncodingAndDecodingMatchTest_LZ4Frame (:132-139): v1 frame of the whole file, checksum verification on."""
    comp, st = oracle.encode(A.FMT_LZ4, bmp, A.make_opts(quality=8))
    assert st == 0 and comp[:4] == bytes([0x04, 0x22, 0x4D, 0x18])
    out, out_len, consumed, status = oracle.decode(A.FMT_LZ4, comp, len(bmp), A.make_opts(lz4_verify=1))
    assert status == 0 and out == bmp


@pytest.mark.parametrize("fmt", [f for f in ALL_FORMATS if f not in (A.FMT_LZ4_BLOCK, A.FMT_SNAPPY_BLOCK, A.FMT_YAZ1)], ids=fmt_id)
def test_data_recognition(oracle, fmt):
    """DataRecognitionTest (:60-80): 256 zero bytes at Fastest; IsMatch true; GetDecompressedSize == 0x100."""
    comp, st = oracle.encode(fmt, bytes(0x100), A.make_opts(quality=0))
    assert st == 0
    assert oracle.is_match(fmt, comp)
    if fmt in SIZED_FORMATS:
        size, st = oracle.decoded_size(fmt, comp)
        assert st == 0 and size == 0x100
    else:
        size, st = oracle.decoded_size(fmt, comp)
        assert st == A.NOT_SUPPORTED
        size, st = oracle.decoded_size(fmt, comp, size_scan=1)
        assert st == 0 and size == 0x100


def test_lz4_block_cross_check_with_system_liblz4(oracle, bmp):
    """Second opinion for the LZ4 block format from liblz4 1.9.4, recorded so that the test needs no system library:
    LZ4_decompress_safe decoded the oracle's block of the first 200 000 bytes of Test.bmp (SHA-256 below) to those bytes, and
    tests/golden/liblz4_block_of_bmp_200000.lz4 is LZ4_compress_default's block of the same bytes."""
    raw = bmp[:200000]
    comp, st = oracle.encode(A.FMT_LZ4_BLOCK, raw, A.make_opts(quality=8))
    assert st == 0 and hashlib.sha256(comp).hexdigest() == "a3479a738b3689a7cc2e01ba541cce0a75d31f44d9180884aa0cd0f9d6fcd79c"
    ref = open(os.path.join(ROOT, "tests", "golden", "liblz4_block_of_bmp_200000.lz4"), "rb").read()
    out, out_len, consumed, status = oracle.decode(A.FMT_LZ4_BLOCK, ref, len(raw))
    assert status == 0 and out == raw


def test_status_taxonomy(oracle, bmp):
    comp, _ = oracle.encode(A.FMT_LZ10, bmp[:5000], A.make_opts(quality=8))
    assert oracle.decode(A.FMT_LZ10, comp[:100], 5000)[3] == A.END_OF_STREAM
    assert oracle.decode(A.FMT_LZ10, b"\x11" + comp[1:], 5000)[3] == A.INVALID_IDENTIFIER
    assert oracle.decode(A.FMT_LZ10, comp, 4999)[3] == A.DST_TOO_SMALL
    short = bytearray(comp)
    short[1:4] = (4990).to_bytes(3, "little")          # header claims fewer bytes than the tokens produce
    assert oracle.decode(A.FMT_LZ10, bytes(short), 6000)[3] in (A.SIZE_MISMATCH, A.OK)
    yaz, _ = oracle.encode(A.FMT_YAZ0, bmp[:5000], A.make_opts(quality=8, byte_order=A.ENDIAN_LITTLE))
    out, out_len, consumed, status = oracle.decode(A.FMT_YAZ0, yaz, 1 << 20)      # default Big: the swapped-size retry decodes it
    assert status == 0 and out == bmp[:5000]
    dict_frame = (0x184D2204).to_bytes(4, "little") + bytes([0x41, 0x40]) + b"\x01\x02\x03\x04\x00"
    assert oracle.decode(A.FMT_LZ4, dict_frame, 100)[3] == A.NOT_SUPPORTED
    assert oracle.decode(A.FMT_SNAPPY, bytes([0xff, 6, 0, 0]) + b"sNaPpY" + bytes([5, 1, 0, 0, 9]), 100)[3] == A.INVALID_DATA


def test_ragged_and_empty_inputs(oracle):
    rng = np.random.default_rng(7)
    for fmt in ALL_FORMATS:
        raws = [synth(rng, n, k) for k, n in enumerate([0, 1, 2, 3, 4, 5, 6, 15, 16, 17, 4096, 4097, 70000])]
        comps, st = oracle.encode_batch(fmt, raws, A.make_opts(quality=8), threads=2)
        outs, out_len, consumed, dst = oracle.decode_batch(fmt, comps, [len(r) for r in raws], threads=2)
        for r, s, o, d in zip(raws, st, outs, dst):
            if s == 0 and d == 0:
                assert o == r
            else:   # the reference's own quirks: LZ4 block encoders reject < 5 bytes; empty LZ10/LZ11/LZ4Legacy/LZO do not
                # decode; PRS's byte-order heuristic (PRS.cs:161-218) misfires on high-entropy data
                assert len(r) < 5 or fmt == A.FMT_PRS


def test_reference_lzo_encoder_back_to_back_literal_runs(oracle):
    """A quirk of the reference's LZO encoder that the oracle (and the GPU encoder) reproduce: LZO.cs:168-176 shortens a match
    that starts fewer than 4 bytes behind the cursor so that the literal run in front of it is 4 bytes long, and when
    fewer than MinLength bytes of the match are left (:188) nothing is written for it — the next token is then a second
    literal run, which LZO1X cannot express after a run (the decoder, :71-86, takes its flag for a 3-byte match at distance
    > 2048).  Such a stream does not round-trip through the reference; the bar for it is decoder parity (tests/
    test_baseline_sizes_gpu.py), and the bench's LZO line leaves these streams out and says how many."""
    raw = bytes([247, 7] * 3 + [252, 13] * 40 + list(range(50)))
    enc, st = oracle.encode(A.FMT_LZO, raw, A.make_opts(quality=8))
    assert st == 0 and enc[:6] == bytes([0x01, 247, 7, 247, 7, 0x01])   # 4 literals, then ANOTHER literal-run flag
    out, out_len, consumed, status = oracle.decode(A.FMT_LZO, enc, len(raw) + 64)
    assert status == 0 and out_len != len(raw) and out[:len(raw)] != raw
