"""Wrapper formats (SURVEY.md 8f item 2): GCLZ, CXLZ, COMP, 3DS-LZ, LZ77 (LZ10 / LZ11 / ChunkLZ10), Level5 (stored / LZ10),
LZOn, Level5LZSS — a header around a core the kernels decode.

CPU part (not gpu): the oracle's restatement against hand-derived layouts (the reference holds no golden vector for these
formats: parity unpinned beyond the cores they wrap).  GPU part: byte-exact parity of libaurora_cuda.so with the oracle on
valid, truncated and corrupt inputs, encoder parity, and the Python mirror of the reference's classes."""
import io

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests.util import corrupt, fmt_id, literal_lzss0_body, lz00_file, lz00_stream, lz00_stream_fast, synth

WRAPPERS = A.WRAPPER_FORMATS
NO_IDENTIFIER = (A.FMT_LEVEL5, A.FMT_LZSEGA, A.FMT_GCZ)   # no magic: IsMatch is a heuristic on zlib / lengths / the file name
LZON_MAGIC = b"LZOn\x00\x2f\xf1\x71"


def _opt_sets(fmt):
    if fmt == A.FMT_LZ77:
        return [dict(), dict(lz77_type=0x11), dict(lz77_type=0xF7), dict(lz77_type=0xF7, lz77_chunk_size=0x400)]
    if fmt == A.FMT_LEVEL5:
        return [dict(), dict(quality=0)]
    if fmt == A.FMT_ECD:
        return [dict(), dict(quality=0), dict(ecd_plain_size=9)]
    if fmt == A.FMT_LZ00:
        return [dict(), dict(lz00_key=0xDEADBEEF)]
    return [dict()]


# ------------------------------------------------------------------------------------------------ CPU: oracle layouts
def test_oracle_wrapper_layouts(oracle, bmp):
    raw = bmp[:20000]
    q8 = A.make_opts(quality=8)
    lz10, _ = oracle.encode(A.FMT_LZ10, raw, q8)
    lz11, _ = oracle.encode(A.FMT_LZ11, raw, q8)
    lzo, _ = oracle.encode(A.FMT_LZO, raw, q8)
    enc = lambda f, **kw: oracle.encode(f, raw, A.make_opts(**({"quality": 8} | kw)))[0]
    assert enc(A.FMT_GCLZ) == b"GCLZ" + lz10            # GCLZ.cs:41-45
    assert enc(A.FMT_CXLZ) == b"CXLZ" + lz10            # CXLZ.cs:43-47
    assert enc(A.FMT_COMP) == b"COMP" + lz11            # COMP.cs:41-45
    assert enc(A.FMT_LZ_3DS) == b"3DS-LZ\r\n" + lz10    # 3DS-LZ.cs:45-50
    assert enc(A.FMT_LZ77) == b"LZ77" + lz10            # LZ77.cs:59-105, Type LZ10
    assert enc(A.FMT_LZ77, lz77_type=0x11) == b"LZ77" + lz11
    # Level5.cs:127: (int)Type | (length << 3), then the headerless LZ10 body (LZ10's own header is 4 bytes here)
    assert enc(A.FMT_LEVEL5) == (1 | (len(raw) << 3)).to_bytes(4, "little") + lz10[4:]
    assert enc(A.FMT_LEVEL5, quality=0) == (len(raw) << 3).to_bytes(4, "little") + raw   # quality 0 stores (:121-122)
    # LZOn.cs:64-79: identifier, BE size, BE compressed size
    assert enc(A.FMT_LZON) == LZON_MAGIC + len(raw).to_bytes(4, "big") + len(lzo).to_bytes(4, "big") + lzo
    # Level5LZSS.cs:60-72: "SSZL", 0, compressed size, size (LE) + LZSS body with Lzss0Properties (0x1000, 18, 3, 0xFEE)
    lzss0, _ = oracle.encode(A.FMT_LZSS, raw, A.make_opts(quality=8, lzss=A.lz_props_window(0x1000, 0xF + 3, 3, 0xFEE)))
    assert enc(A.FMT_LEVEL5_LZSS) == b"SSZL" + bytes(4) + (len(lzss0) - 16).to_bytes(4, "little") + len(raw).to_bytes(4, "little") + lzss0[16:]
    # the LZSS-property family: fixed headers around the headerless LZSS body (Default (12,4,2) or Lzss0 properties)
    lzssd, _ = oracle.encode(A.FMT_LZSS, raw, q8)
    bd, b0, n = lzssd[16:], lzss0[16:], len(raw)
    le = lambda v: v.to_bytes(4, "little")
    assert enc(A.FMT_AKLZ) == b"AKLZ~?Qd=\xcc\xcc\xcd" + n.to_bytes(4, "big") + bd                       # AKLZ.cs:51-56
    assert enc(A.FMT_LZ01) == b"LZ01" + le(16 + len(b0)) + le(n) + le(0) + b0                                # LZ01.cs:65-82
    assert enc(A.FMT_FCMP) == b"FCMP" + le(n) + le(305397760) + b0                                           # FCMP.cs:52-59
    assert enc(A.FMT_IECP) == b"IECP" + le(n) + b0                                                           # IECP.cs:50-55
    assert enc(A.FMT_MDB4) == b"MDB4" + le(n + 1) + le(n) + le(16 + len(bd)) + bytes(16) + bd                # MDB4.cs:61-80
    assert enc(A.FMT_LZSEGA) == le(len(bd)) + le(n) + bd                                                     # LZSega.cs:57-67
    assert enc(A.FMT_GCZ) == le(n) + b0                                                                      # GCZ.cs:47-51
    assert enc(A.FMT_SDPC) == b"SDPC" + le(n) + lzo                                                          # SDPC.cs:59-64
    # ECD.cs:88-121: "ECD", flag, BE plain size / compressed size (plain bytes + body) / size, 4 plain bytes, LZSS body of
    # the rest with LzProperties(0x400, 0x42, 3, 0x3BE); quality 0 and incompressible inputs are stored
    ecd_body = oracle.encode(A.FMT_LZSS, raw[4:], A.make_opts(quality=8, lzss=A.lz_props_window(0x400, 0x42, 3, 0x3BE)))[0][16:]
    be = lambda v: v.to_bytes(4, "big")
    assert enc(A.FMT_ECD) == b"ECD\x01" + be(4) + be(4 + len(ecd_body)) + be(n) + raw[:4] + ecd_body
    assert enc(A.FMT_ECD, quality=0) == b"ECD\x00" + be(0) + be(n) + be(n) + raw
    noise = bytes(np.random.default_rng(5).integers(0, 256, 3000, dtype=np.uint8))
    assert oracle.encode(A.FMT_ECD, noise, q8)[0] == b"ECD\x00" + be(0) + be(3000) + be(3000) + noise
    assert oracle.encode(A.FMT_ECD, raw[:16], q8)[0] == b"ECD\x00" + be(0) + be(16) + be(16) + raw[:16]   # Length > 0x10 compresses
    # LZ00.cs:83-139: 64-byte header, then the Lzss0 body XORed byte by byte with lz00_stream (the reference's ladder, literally)
    key = 0x5EEDC0DE
    z = enc(A.FMT_LZ00, lz00_key=key)
    assert z[:64] == b"LZ00" + le(64 + len(b0)) + bytes(8) + b"Temp.dat" + bytes(24) + le(n) + le(key) + bytes(8)
    assert z[64:] == bytes(a ^ b for a, b in zip(b0, lz00_stream(key, len(b0))))
    # ChunkLZ10 (LZ77.cs:75-100): 0xF7 | size << 8, u16 end offsets, independent LZ10 streams of ChunkSize bytes
    ch = enc(A.FMT_LZ77, lz77_type=0xF7)
    nseg = (len(raw) + 0xFFF) // 0x1000
    assert ch[:8] == b"LZ77" + (0xF7 | (len(raw) << 8)).to_bytes(4, "little")
    ends = [int.from_bytes(ch[8 + 2 * k:10 + 2 * k], "little") for k in range(nseg)]
    body = 8 + 2 * nseg
    start = 0
    for k in range(nseg):
        piece, _ = oracle.encode(A.FMT_LZ10, raw[k * 0x1000:(k + 1) * 0x1000], q8)
        assert ch[body + start:body + ends[k]] == piece
        start = ends[k]
    assert body + ends[-1] == len(ch)
    # a source that fits one chunk is a plain LZ10 stream (:75)
    assert oracle.encode(A.FMT_LZ77, raw[:100], A.make_opts(quality=8, lz77_type=0xF7))[0] == b"LZ77" + oracle.encode(A.FMT_LZ10, raw[:100], q8)[0]


@pytest.mark.parametrize("fmt", WRAPPERS, ids=fmt_id)
def test_oracle_wrapper_roundtrip_and_errors(oracle, bmp, fmt):
    rng = np.random.default_rng(7000 + fmt)
    for kw in _opt_sets(fmt):
        opts = A.make_opts(**({"quality": 8} | kw))
        for n in (1, 5, 100, 4096, 4097, 20000, 70000):
            raw = synth(rng, n, n % 5)
            c, st = oracle.encode(fmt, raw, opts)
            assert st == 0
            outs, olen, cons, dst = oracle.decode_batch(fmt, [c], [n], opts)
            if fmt in (A.FMT_LZON, A.FMT_SDPC) and not (dst[0] == 0 and outs[0] == raw):
                continue   # the LZO encoder's dropped-first-match quirk (DESIGN.md section 2)
            assert dst[0] == 0 and outs[0] == raw and cons[0] == len(c), (fmt_id(fmt), kw, n, dst[0])
            assert oracle.decoded_size(fmt, c, opts) == (n, 0)
            if fmt not in NO_IDENTIFIER + (A.FMT_GCLZ, A.FMT_CXLZ, A.FMT_COMP) and len(c) > 0x11:
                assert oracle.is_match(fmt, c, opts)   # (GCLZ / CXLZ / COMP add the LZ10 / LZ11 token-walk heuristic)
    # wrong identifier / truncated header
    c, _ = oracle.encode(fmt, bmp[:3000], A.make_opts(quality=8))
    if fmt not in NO_IDENTIFIER:
        bad = b"XXXX" + c[4:]
        _, _, cons, dst = oracle.decode_batch(fmt, [bad], [3000])
        assert dst[0] == A.INVALID_IDENTIFIER
    _, _, cons, dst = oracle.decode_batch(fmt, [c[:3]], [3000])
    assert dst[0] == A.END_OF_STREAM and cons[0] == 3
    _, _, _, dst = oracle.decode_batch(fmt, [c], [2999])
    assert dst[0] == A.DST_TOO_SMALL


def test_lz00_keystream_restatements_agree():
    """lz00_stream_fast (block-wise affine jumps) gives lz00_stream's bytes (the reference's ladder) for every key and length"""
    rng = np.random.default_rng(32)
    for key in [0, 1, 0xFFFFFFFF, 0x5EEDC0DE] + [int(k) for k in rng.integers(0, 1 << 32, size=4)]:
        for count in (0, 1, 255, 256, 257, 511, 513, 3000):
            assert lz00_stream_fast(key, count) == lz00_stream(key, count), (hex(key), count)


def test_oracle_decodes_hand_built_lz00_files(oracle):
    """the literal-only LZ00 files the keystream tests build: every body length except 1 mod 9, decoded by the oracle"""
    rng = np.random.default_rng(33)
    for n in (0, 1, 7, 8, 9, 100, 2047, 8191):
        raw = rng.integers(0, 256, size=n, dtype=np.uint8).tobytes()
        body = literal_lzss0_body(raw)
        assert len(body) == n + (n + 7) // 8
        z = lz00_file(body, n, 0xC0FFEE + n)
        outs, olen, cons, st = oracle.decode_batch(A.FMT_LZ00, [z], [n])
        assert st[0] == A.OK and outs[0] == raw and cons[0] == len(z)


def test_oracle_unsupported_subtypes(oracle):
    """Huffman / RLE / zlib payloads of LZ77 and Level5 are outside the LZ hot path: NOT_SUPPORTED (oracle and GPU agree)."""
    for blob in (b"LZ77" + bytes([0x28, 4, 0, 0]) + bytes(16), b"LZ77" + bytes([0x30, 4, 0, 0]) + bytes(16)):
        assert oracle.decode_batch(A.FMT_LZ77, [blob], [64])[3][0] == A.NOT_SUPPORTED
    assert oracle.decode_batch(A.FMT_LEVEL5, [(2 | (16 << 3)).to_bytes(4, "little") + bytes(16)], [64])[3][0] == A.NOT_SUPPORTED
    assert oracle.decode_batch(A.FMT_LEVEL5, [(64).to_bytes(4, "little") + b"\x78\x9c" + bytes(16)], [64])[3][0] == A.NOT_SUPPORTED


# ------------------------------------------------------------------------------------------------ GPU: parity
def _compare(codec, oracle, fmt, comps, caps, opts=None, what=""):
    outs, out_len, consumed, status = codec.decode_batch(fmt, comps, caps, opts)
    ref, rlen, rcons, rst = oracle.decode_batch(fmt, comps, caps, opts)
    bad = [i for i in range(len(comps)) if status[i] != rst[i] or out_len[i] != rlen[i] or consumed[i] != rcons[i] or outs[i] != ref[i]]
    if bad:
        i = bad[0]
        pytest.fail(f"{fmt_id(fmt)} {what}: {len(bad)}/{len(comps)} streams differ; first #{i}: status gpu={status[i]} ref={rst[i]}, "
                    f"out_len {out_len[i]}/{rlen[i]}, consumed {consumed[i]}/{rcons[i]}, srclen {len(comps[i])}, cap {caps[i]}")
    return outs, status


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", WRAPPERS, ids=fmt_id)
def test_gpu_wrapper_decode_parity(codec, oracle, fmt):
    rng = np.random.default_rng(8000 + fmt)
    for kw in _opt_sets(fmt):
        opts = A.make_opts(**({"quality": 8} | kw))
        raws = [synth(rng, int(rng.choice([1, 2, 7, 100, 1000, 4095, 4096, 4097, 9000, 40000, 70000])), i % 5) for i in range(60)]
        comps, st = oracle.encode_batch(fmt, raws, opts)
        # ChunkLZ10 refuses inputs whose chunks end past 0xFFFF ("chunks too large to process", LZ77.cs:93-96)
        assert (st == 0).all() or kw.get("lz77_type") == 0xF7
        raws = [r for r, s_ in zip(raws, st) if s_ == 0]
        comps = [c for c, s_ in zip(comps, st) if s_ == 0]
        outs, status = _compare(codec, oracle, fmt, comps, [len(r) for r in raws], opts, what=f"valid {kw}")
        ok = sum(1 for i, r in enumerate(raws) if status[i] == 0 and outs[i] == r)
        assert ok >= len(raws) - (6 if fmt in (A.FMT_LZON, A.FMT_SDPC) else 0)
        # truncated / bit-flipped / padded / empty / header-cut inputs, and short destinations
        bad = [corrupt(rng, c, i % 5) for i, c in enumerate(comps)]
        _compare(codec, oracle, fmt, bad, [len(r) + int(rng.choice([0, 0, 64])) for r in raws], opts, what=f"fuzz {kw}")
        _compare(codec, oracle, fmt, comps, [max(0, len(r) + int(rng.choice([-len(r), -17, -1, 0, 1, 100]))) for r in raws], opts, what=f"capacity {kw}")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", [A.FMT_LEVEL5, A.FMT_ECD], ids=fmt_id)
def test_gpu_wrapper_mixed_stored_and_compressed(codec, oracle, fmt):
    """Stored payloads / ECD's plain prefix are written by the host; they must survive the core batch's device-to-host copy
    of the destination span when stored and compressed streams alternate in ONE batch."""
    rng = np.random.default_rng(8500 + fmt)
    raws = [synth(rng, int(rng.choice([17, 100, 3000, 20000])), i % 5) for i in range(40)]
    comps = [oracle.encode(fmt, r, A.make_opts(quality=0 if i % 2 else 8))[0] for i, r in enumerate(raws)]
    outs, status = _compare(codec, oracle, fmt, comps, [len(r) for r in raws], what="mixed")
    assert (status == 0).all() and all(o == r for o, r in zip(outs, raws))


@pytest.mark.gpu
def test_gpu_wrapper_unsupported_subtypes(codec, oracle):
    blobs = [b"LZ77" + bytes([0x28, 4, 0, 0]) + bytes(16), b"LZ77" + bytes([0x30, 4, 0, 0]) + bytes(16), b"LZ77" + bytes([0x42, 4, 0, 0]) + bytes(16)]
    _compare(codec, oracle, A.FMT_LZ77, blobs, [64] * 3, what="lz77 subtypes")
    blobs = [(2 | (16 << 3)).to_bytes(4, "little") + bytes(16), (64).to_bytes(4, "little") + b"\x78\x9c" + bytes(16), bytes(4), bytes(5)]
    _compare(codec, oracle, A.FMT_LEVEL5, blobs, [64] * 4, what="level5 subtypes")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", WRAPPERS, ids=fmt_id)
def test_gpu_wrapper_encode_parity(codec, oracle, fmt):
    rng = np.random.default_rng(9000 + fmt)
    for kw in _opt_sets(fmt):
        opts = A.make_opts(**({"quality": 8} | kw))
        raws = [synth(rng, int(rng.choice([1, 5, 6, 100, 4096, 4097, 12000, 30000])), i % 5) for i in range(24)]
        got, st = codec.encode_batch(fmt, raws, opts)
        ref, rst = oracle.encode_batch(fmt, raws, opts)
        assert (st == rst).all() and ((st == 0).all() or kw.get("lz77_type") == 0xF7), (fmt_id(fmt), kw, st, rst)
        keep = [i for i in range(len(raws)) if st[i] == 0]
        raws, got, ref = [raws[i] for i in keep], [got[i] for i in keep], [ref[i] for i in keep]
        bad = [i for i in range(len(raws)) if got[i] != ref[i]]
        assert not bad, f"{fmt_id(fmt)} {kw}: {len(bad)} streams differ from the oracle encoder, first #{bad[0]} ({len(raws[bad[0]])} bytes)"
        size, sst = codec.decoded_size_batch(fmt, got, opts)
        assert (sst == 0).all() and [int(x) for x in size] == [len(r) for r in raws]
        if fmt not in NO_IDENTIFIER:
            m = codec.is_match_batch(fmt, got, opts)
            assert [bool(x) for x in m] == [bool(oracle.is_match(fmt, g, opts)) for g in got]


@pytest.mark.gpu
def test_gpu_wrapper_mirror_classes(bmp):
    """The reference-facing classes: Compress / Decompress / GetDecompressedSize / IsMatch over streams."""
    from auroralib.compression_b200 import (AKLZ, COMP, CXLZ, ECD, FCMP, GCLZ, GCZ, IECP, LZ00, LZ01, LZ77, LZ_3DS, MDB4, CompressionSettings,
                                            InvalidIdentifierException, Level5, Level5LZSS, LZOn, LZSega, SDPC)
    raw = bmp[:30000]
    for cls in (GCLZ, CXLZ, COMP, LZ_3DS, LZ77, Level5, LZOn, Level5LZSS, AKLZ, LZ01, FCMP, IECP, MDB4, LZSega, GCZ, SDPC, ECD, LZ00):
        alg = cls()
        blob = alg.Compress(raw, settings=CompressionSettings(8)).getvalue()
        src = io.BytesIO(b"pad" + blob + b"tail")
        src.seek(3)
        assert alg.GetDecompressedSize(src) == len(raw) and src.tell() == 3
        dst = io.BytesIO()
        alg.Decompress(src, dst)
        assert dst.getvalue() == raw and src.tell() == 3 + len(blob)
        if cls not in (Level5, LZSega, GCZ):
            assert alg.IsMatch(io.BytesIO(blob)) and not alg.IsMatch(io.BytesIO(b"nope" + blob[4:]))
            with pytest.raises(InvalidIdentifierException):
                alg.Decompress(io.BytesIO(b"nope" + blob[4:]), io.BytesIO())
    # LZ00.Compress(source, destination, key, settings) and ECD.PlainSize
    z = LZ00().Compress(raw, key=0x1234, settings=CompressionSettings(8)).getvalue()
    assert z[52:56] == (0x1234).to_bytes(4, "little") and LZ00().Decompress(io.BytesIO(z)).getvalue() == raw
    e = ECD()
    e.PlainSize = 11
    z = e.Compress(raw, settings=CompressionSettings(8)).getvalue()
    assert z[4:8] == (11).to_bytes(4, "big") and z[16:27] == raw[:11] and ECD().Decompress(io.BytesIO(z)).getvalue() == raw
    assert ECD().Decompress(io.BytesIO(ECD().Compress(raw, settings=CompressionSettings(0)).getvalue())).getvalue() == raw
    chunked = LZ77()
    chunked.Type, chunked.ChunkSize = LZ77.CHUNK_LZ10_TYPE, 0x800
    blob = chunked.Compress(raw, settings=CompressionSettings(8)).getvalue()
    assert blob[4] == 0xF7 and LZ77().Decompress(io.BytesIO(blob)).getvalue() == raw


@pytest.mark.gpu
def test_lz77_mixed_sub_types_in_one_batch(codec, oracle, bmp):
    """ADVICE round 1: a wrapped batch that needs more than one core batch (LZ77 resolves type 0x10 to LZ10, 0x11 to LZ11 and 0xF7
    to ChunkLZ10) runs several core batches over ONE destination; every stream must keep the bytes its own core batch decoded,
    also when two chunked files fail and are decoded once more."""
    rng = np.random.default_rng(77)
    raws = [bmp[int(o):int(o) + int(n)] for o, n in zip(rng.integers(0, 900000, size=90), rng.integers(200, 30000, size=90))]
    types = [(0x10, 0), (0x11, 0), (0xF7, 0), (0xF7, 0x400)]
    comps = []
    for i, r in enumerate(raws):
        t, cs = types[i % 4]
        c, st = oracle.encode(A.FMT_LZ77, r, A.make_opts(quality=8, lz77_type=t, lz77_chunk_size=cs))
        assert st == 0
        comps.append(c)
    # two chunked files that fail: cut inside their last chunk
    for k in (2, 6):
        comps[k] = comps[k][:len(comps[k]) - 40]
    caps = [len(r) for r in raws]
    outs, out_len, consumed, status = codec.decode_batch(A.FMT_LZ77, comps, caps)
    ref, rlen, rcons, rst = oracle.decode_batch(A.FMT_LZ77, comps, caps)
    assert (status == rst).all() and (out_len == rlen).all() and (consumed == rcons).all()
    assert outs == ref
    assert sum(1 for i in range(len(raws)) if status[i] == 0 and outs[i] == raws[i]) == len(raws) - 2
