"""The kernels' DEVICE SOURCE on a CPU lane emulation (tests/simt/: one fiber per lane, warp primitives and named barriers as
rendezvous points, bounds-checked shared memory, a synchronous checked TMA), compared with the oracle.  The device part of each
real kernel file (everything above its "// ---- kernel" line) is compiled by g++ against stand-in headers:
  * encoders — csrc/encode_lz_par.cu (one lane per window position) and csrc/encode_lz.cu / encode_bytelz.cu with finder.cuh (the
    sequential replay): every format and quality, the small-match table, matches beyond the data ring's lookahead, the
    three-section writers, CompatibilityMode, unaligned sources, too-small destinations;
  * decoders — csrc/decode_flaglz.cu (the headline kernel: a parser warp and a resolver warp per stream slot), decode_bytelz.cu,
    decode_blz.cu: valid and corrupt streams, exact / short / larger destinations; status, out_len, consumed and bytes;
  * the IsMatch and GetDecompressedSize rules of csrc/ismatch.cu (plain per-stream functions, no lanes): every matchable format
    on streams, corrupted streams, raw data and every offset of a ROM-like image.
No GPU: this is the check of the kernels' lane-level logic that runs in the CPU suite, on more inputs than GPU time allows."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests.util import MATCHABLE, SIZED_FORMATS, decoded_size_blobs, fmt_id, is_match_blobs, rom_like_image, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIMT = os.path.join(ROOT, "tests", "simt")
CSRC = os.path.join(ROOT, "auroralib", "compression_b200", "csrc")
PAR_FORMATS = [A.FMT_LZ10, A.FMT_BLZ, A.FMT_YAZ0, A.FMT_YAZ1, A.FMT_LZSS, A.FMT_MIO0, A.FMT_YAY0, A.FMT_LZ11, A.FMT_LZ40, A.FMT_LZ60,
               A.FMT_LZHUDSON, A.FMT_SMSR00]


def _build(name, harness, macro, extra=()):
    build = os.path.join(SIMT, "build")
    os.makedirs(build, exist_ok=True)
    src = open(os.path.join(CSRC, name + ".cu")).read()
    inc = os.path.join(build, name + "_device.inc")
    with open(inc, "w") as f:
        f.write(src[:src.index("// ---- kernel\n")])   # the device functions; the kernel entry and the launcher stay out
    so = os.path.join(build, f"libsimt_{name}.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", SIMT, "-I", CSRC,
                           f'-DAURORA_REAL_COMMON="{os.path.join(CSRC, "common.cuh")}"', f'-DAURORA_REAL_STAGE="{os.path.join(CSRC, "stage.cuh")}"',
                           f'-D{macro}="{inc}"', *extra,
                           os.path.join(SIMT, harness), "-o", so])
    return C.CDLL(so)


class SimtLibs:
    def __init__(self):
        self.par = _build("encode_lz_par", "par_harness.cpp", "PAR_DEVICE_INC").simt_encode_lz_par
        self.seq_flag = _build("encode_lz", "seq_harness.cpp", "SEQ_DEVICE_INC").simt_encode_seq
        self.seq_byte = _build("encode_bytelz", "seq_harness.cpp", "SEQ_DEVICE_INC", ["-DSEQ_BYTELZ"]).simt_encode_seq
        for f in (self.par, self.seq_flag, self.seq_byte):
            f.restype = C.c_int


@pytest.fixture(scope="session")
def simt_lib():
    return SimtLibs()


BYTE_FORMATS = [A.FMT_LZ4, A.FMT_LZ4_LEGACY, A.FMT_LZ4_BLOCK, A.FMT_LZO, A.FMT_SNAPPY, A.FMT_SNAPPY_BLOCK, A.FMT_PRS]
SEQ_FLAG_FORMATS = PAR_FORMATS


def _isqrt2q(q):
    r = 0
    while (r + 1) * (r + 1) <= 2 * q:
        r += 1
    return r


def finder_params(fmt, quality, strategy=0, vram_mode=-1, lzss=None):
    """CompressionSettings + LzProperties -> LzChainMatchFinder parameters (LzChainMatchFinder.cs:42-119), as api.cu
    fill_encode_params derives them."""
    if fmt == A.FMT_LZ10:
        lz = A.lz_props_window(0x1000, 18, 3, 0, 2 if vram_mode != 0 else 1)
    elif fmt == A.FMT_BLZ:
        lz = A.lz_props_window(0x1000, 18, 3, 0, 3)
    elif fmt in (A.FMT_LZ11, A.FMT_LZ40, A.FMT_LZ60):
        lz = A.lz_props_window(0x1000, 0x4000, 3, 0, 2 if vram_mode > 0 else 1)
    elif fmt in (A.FMT_YAZ0, A.FMT_YAZ1, A.FMT_YAY0, A.FMT_LZHUDSON):
        lz = A.lz_props_window(0x1000, 0xFF + 0x12, 3, 0, 1)
    elif fmt in (A.FMT_MIO0, A.FMT_SMSR00):
        lz = A.lz_props_window(0x1000, 18, 3, 0, 1)
    elif fmt in (A.FMT_LZ4, A.FMT_LZ4_LEGACY, A.FMT_LZ4_BLOCK):
        lz = A.lz_props_window(0xFFFF, 0x7FFFFFFF, 4, 0, 1)
    elif fmt == A.FMT_LZO:
        lz = A.lz_props_window(0xBFFF, 0x7FFFFFFF, 3, 0, 1)
    elif fmt in (A.FMT_SNAPPY, A.FMT_SNAPPY_BLOCK):
        lz = A.lz_props_window(0x8000, 64, 4, 0, 1)
    elif fmt == A.FMT_PRS:
        lz = A.lz_props_window(0x1FFF, 0x100, 2, 0, 1)
    else:
        lz = lzss if lzss is not None else A.lz_props_bits(12, 4, 2)
    q = quality
    max_chain = q + 1 if q < 6 else 1 << (q - 5) if q >= 11 else (1 << (q >> 1)) | ((1 << (q >> 1)) >> (q & 1))
    finder = [max_chain, 3 + q // 3, 15 + _isqrt2q(q), min(17 + _isqrt2q(q), max(1, lz.windows_bits)), lz.min_length, lz.max_length,
              lz.min_distance, lz.max_distance, strategy & 1, 1 if q >= 10 else 0]
    return finder, [lz.windows_bits, lz.length_bits, lz.min_length, lz.max_distance, lz.windows_start]


def simt_encode(lib, fmt, raws, quality, strategy=0, byte_order=A.ENDIAN_DEFAULT, vram_mode=-1, lzss=None, yaz0_alignment=0,
                caps=None, skew=0, seq=False, lz4_block_size=0):
    """One emulated warp encodes `raws`: the lane-per-position search, or (seq) the sequential replay of finder.cuh."""
    n = len(raws)
    finder, lzp = finder_params(fmt, quality, strategy, vram_mode, lzss)
    # sources back to back from an odd offset (any alignment is allowed), readable up to the next multiple of 16
    off, pos = [], skew
    for r in raws:
        off.append(pos)
        pos += len(r) + (pos % 3)
    limit = (pos + 15) & ~15
    backing = np.zeros(limit + 64, dtype=np.uint8)
    a0 = (-backing.ctypes.data) % 16
    src = backing[a0:a0 + limit]
    for o, r in zip(off, raws):
        src[o:o + len(r)] = np.frombuffer(r, dtype=np.uint8)
    if caps is None:
        caps = [len(r) + len(r) // 6 + 256 for r in raws]
    doff, dpos = [], 0
    for c in caps:
        doff.append(dpos)
        dpos += c + 8
    dst = np.full(dpos + 8, 0xEE, dtype=np.uint8)
    longest = max([len(r) for r in raws] + [0])
    spw = 2 * (longest + 64) + 256
    if seq:   # csrc/encode_lz.cu encode_scratch_per_warp: head + chain + small-match tables in front of the section staging
        spw = ((4 << finder[2]) + (4 << finder[3]) + 65536 * 4 + 2 * (longest + 64) + 255) & ~255
    backing_s = np.full(spw + 128, 0xEE, dtype=np.uint8)
    s0 = (-backing_s.ctypes.data) % 16
    scratch = backing_s[s0:s0 + spw + 64]
    out_len = np.zeros(n, dtype=np.uint64)
    status = np.full(n, 77, dtype=np.int32)
    u64 = lambda v: np.asarray(v, dtype=np.uint64)
    src_off, src_len, dst_off, dst_cap = u64(off), u64([len(r) for r in raws]), u64(doff), u64(caps)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    tail = (p(src), C.c_uint64(limit), p(src_off), p(src_len), p(dst), p(dst_off), p(dst_cap), p(out_len), p(status), C.c_uint32(n),
            p(scratch), C.c_uint64(spw))
    head = (C.c_int(fmt), C.c_int(byte_order), (C.c_int * 10)(*finder), C.c_uint32(yaz0_alignment))
    if seq:
        entry = lib.seq_byte if fmt in BYTE_FORMATS else lib.seq_flag
        rc = entry(*head, C.c_uint32(lz4_block_size or 0x400000), (C.c_int * 5)(*lzp), *tail)
    else:
        rc = lib.par(*head, (C.c_int * 5)(*lzp), *tail)
    assert rc == 0
    assert (scratch[spw:] == 0xEE).all(), "the section staging ran over its slice of the scratch buffer"
    outs = []
    for i in range(n):
        assert (dst[doff[i] + caps[i]:doff[i] + caps[i] + 8] == 0xEE).all(), f"stream {i}: bytes written past the capacity"
        outs.append(dst[doff[i]:doff[i] + min(int(out_len[i]), caps[i])].tobytes())
    return outs, status, out_len


def _check(lib, oracle, fmt, raws, quality, **kw):
    okw = {k: v for k, v in kw.items() if k not in ("skew", "seq")}
    ref, rst = oracle.encode_batch(fmt, raws, A.make_opts(quality=quality, **okw))
    if fmt == A.FMT_BLZ:
        # BLZ.cs:143-215: the kernel writes the token body of the REVERSED source (LZ10's layout, distance - 3); the host side
        # reverses that body and appends padding + footer (api.cu), so the reference's stream starts with the reversed body
        got, st, _ = simt_encode(lib, fmt, [r[::-1] for r in raws], quality, **kw)
        assert (st == 0).all()
        ref = [x if len(r) else b"" for x, r in zip(ref, raws)]
        bad = [i for i in range(len(raws)) if rst[i] == 0 and not (ref[i].startswith(got[i][::-1]) and len(ref[i]) - len(got[i]) <= 24)]
    else:
        got, st, _ = simt_encode(lib, fmt, raws, quality, **kw)
        assert (st == rst).all(), (fmt_id(fmt), quality, st, rst)
        bad = [i for i in range(len(raws)) if rst[i] == 0 and got[i] != ref[i]]   # (a failed stream's bytes are unspecified)
    assert not bad, f"{fmt_id(fmt)} q{quality}: stream #{bad[0]} (len {len(raws[bad[0]])}) differs from the oracle encoder: {len(got[bad[0]])} vs {len(ref[bad[0]])} bytes"


@pytest.mark.parametrize("fmt", PAR_FORMATS, ids=fmt_id)
@pytest.mark.parametrize("quality", [0, 3, 8, 10, 15])
def test_kernel_source_on_emulated_lanes(simt_lib, oracle, bmp, fmt, quality):
    rng = np.random.default_rng(31 * fmt + quality)
    raws = [bmp[:n] for n in (5, 33, 4097, 9000)] + [synth(rng, int(n), i % 5) for i, n in enumerate([0, 1, 4, 31, 32, 33, 64, 65, 1000, 4096, 6000, 12000])]
    _check(simt_lib, oracle, fmt, raws, quality, skew=int(rng.integers(0, 16)))
    _check(simt_lib, oracle, fmt, raws[3:12], quality, strategy=A.STRATEGY_COMPATIBILITY, skew=int(rng.integers(0, 16)))


@pytest.mark.parametrize("fmt", [A.FMT_LZ11, A.FMT_LZ40, A.FMT_LZ60], ids=fmt_id)
@pytest.mark.parametrize("quality", [2, 11])
def test_matches_beyond_the_ring_lookahead(simt_lib, oracle, bmp, fmt, quality):
    rng = np.random.default_rng(5 + fmt + quality)
    noise = rng.integers(0, 256, size=3000, dtype=np.uint8).tobytes()
    raws = [bytes(40000), b"abcdefg" * 3000, noise[:300] * 60, noise + noise + noise[:1500] + noise, bytes(289), bytes(320),
            b"\x01" * 16384 + b"\x02" * 16390 + b"\x01" * 400, noise[:1000] + bytes(273 + 4) + noise[:999] + bytes(272 + 4) + noise[:17] + bytes(0x4000 + 5)]
    _check(simt_lib, oracle, fmt, raws, quality, skew=3)
    _check(simt_lib, oracle, fmt, [raws[3], raws[4], raws[5]], quality, strategy=A.STRATEGY_COMPATIBILITY)


def test_streams_over_64k_wrap_the_table_positions(simt_lib, oracle, bmp):
    rng = np.random.default_rng(8)
    raws = [bmp[:70000], synth(rng, 140000, 0), synth(rng, 70000, 2)]
    for fmt, q in ((A.FMT_LZ10, 8), (A.FMT_YAZ0, 5), (A.FMT_MIO0, 10), (A.FMT_LZ11, 12)):
        _check(simt_lib, oracle, fmt, raws, q)


def test_options_and_small_destinations(simt_lib, oracle, bmp):
    raws = [bmp[1000:9000], bytes(5000), bmp[:7]]
    for vram in (0, 1):
        _check(simt_lib, oracle, A.FMT_LZ10, raws, 8, vram_mode=vram)
        _check(simt_lib, oracle, A.FMT_LZ11, raws, 10, vram_mode=vram)
    for order in (A.ENDIAN_BIG, A.ENDIAN_LITTLE):
        for fmt in (A.FMT_YAZ0, A.FMT_YAY0, A.FMT_MIO0):
            _check(simt_lib, oracle, fmt, raws, 4, byte_order=order)
    _check(simt_lib, oracle, A.FMT_YAZ0, raws, 4, yaz0_alignment=0x20)
    for props in (A.lz_props_bits(10, 6, 2), A.lz_props_bits(12, 4, 2), A.lz_props_window(0x1000, 18, 3, 0xFEE)):
        _check(simt_lib, oracle, A.FMT_LZSS, raws, 8, lzss=props)
        _check(simt_lib, oracle, A.FMT_LZSS, raws, 12, lzss=props)
    for fmt in PAR_FORMATS:   # a destination of 100 bytes: DST_TOO_SMALL, the needed length reported, nothing written past the capacity
        got, st, out_len = simt_encode(simt_lib, fmt, [bmp[:20000]], 3, caps=[100])
        assert st[0] == A.DST_TOO_SMALL and out_len[0] > 100, fmt_id(fmt)


@pytest.mark.parametrize("fmt", SEQ_FLAG_FORMATS + BYTE_FORMATS, ids=fmt_id)
@pytest.mark.parametrize("quality", [0, 8, 12])
def test_sequential_replay_on_emulated_lanes(simt_lib, oracle, bmp, fmt, quality):
    """finder.cuh with the token writers of encode_lz.cu / encode_bytelz.cu: the finder every format falls back to."""
    rng = np.random.default_rng(17 * fmt + quality)
    raws = [bmp[:n] for n in (5, 33, 4097, 6000)] + [synth(rng, int(n), i % 5) for i, n in enumerate([0, 1, 4, 31, 32, 33, 64, 65, 1000, 4096, 5000, 7000])]
    _check(simt_lib, oracle, fmt, raws, quality, seq=True, skew=int(rng.integers(0, 16)))
    _check(simt_lib, oracle, fmt, raws[3:12], quality, seq=True, strategy=A.STRATEGY_COMPATIBILITY)


# ---- a decoder on the same emulation: Nintendo BLZ (csrc/decode_blz.cu, the one kernel that keeps everything in global memory)
@pytest.fixture(scope="session")
def simt_blz():
    f = _build("decode_blz", "blz_harness.cpp", "BLZ_DEVICE_INC").simt_decode_blz
    f.restype = C.c_int
    return f


def simt_decode_blz(entry, comps, caps):
    n = len(comps)
    off, pos = [], 5
    for c in comps:
        off.append(pos)
        pos += len(c) + 3
    src = np.zeros(pos + 32, dtype=np.uint8)
    for o, c in zip(off, comps):
        src[o:o + len(c)] = np.frombuffer(c, dtype=np.uint8)
    doff, dpos = [], 0
    for c in caps:
        doff.append(dpos)
        dpos += c + 8
    dst = np.full(dpos + 8, 0xEE, dtype=np.uint8)
    out_len, consumed = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint64)
    status = np.full(n, 77, dtype=np.int32)
    u64 = lambda v: np.asarray(v, dtype=np.uint64)
    src_off, src_len, dst_off, dst_cap = u64(off), u64([len(c) for c in comps]), u64(doff), u64(caps)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    entry(p(src), C.c_uint64(len(src)), p(src_off), p(src_len), p(dst), p(dst_off), p(dst_cap), p(out_len), p(consumed), p(status),
          C.c_uint32(n), C.c_int(0))
    outs = []
    for i in range(n):
        assert (dst[doff[i] + caps[i]:doff[i] + caps[i] + 8] == 0xEE).all(), f"stream {i}: bytes written past the capacity"
        outs.append(dst[doff[i]:doff[i] + int(out_len[i])].tobytes() if status[i] == 0 else b"")
    return outs, out_len, consumed, status


def test_blz_decoder_on_emulated_lanes(simt_blz, oracle, bmp):
    from tests.util import corrupt
    rng = np.random.default_rng(2026)
    raws = [bmp[:n] for n in (33, 4097, 9000)] + [synth(rng, int(n), i % 5) for i, n in enumerate([1, 4, 31, 32, 33, 64, 65, 1000, 4096, 6000, 12000])]
    comps, st = oracle.encode_batch(A.FMT_BLZ, raws, A.make_opts(quality=8))
    assert (st == 0).all()
    streams, caps = [], []
    for i, (c, r) in enumerate(zip(comps, raws)):
        streams.append(c)
        caps.append(len(r))
        for mode in range(5):   # truncated, one byte flipped, garbage appended, empty, cut inside the header
            streams.append(corrupt(rng, c, mode))
            caps.append(len(r) if i % 2 else len(r) + 100)
        streams.append(c)       # destination one byte short
        caps.append(max(len(r) - 1, 0))
    ref, rlen, rcons, rst = oracle.decode_batch(A.FMT_BLZ, streams, caps, A.make_opts())
    got, out_len, consumed, status = simt_decode_blz(simt_blz, streams, caps)
    assert (status == rst).all(), [(i, int(status[i]), int(rst[i])) for i in range(len(streams)) if status[i] != rst[i]][:5]
    assert (out_len == rlen).all() and (consumed == rcons).all()
    assert all(g == r for g, r, s in zip(got, ref, rst) if s == 0)
    assert (rst == 0).sum() >= len(raws)


# ---- the byte-LZ decode kernel (csrc/decode_bytelz.cu: LZ4 block / legacy / frame, Snappy block / framed, LZO, PRS) with the real
#      staged input stream of csrc/stage.cuh over an emulated TMA (a checked memcpy that completes at once)
@pytest.fixture(scope="session")
def simt_bytelz_dec():
    f = _build("decode_bytelz", "bytelz_dec_harness.cpp", "DEC_DEVICE_INC").simt_decode_bytelz
    f.restype = C.c_int
    return f


def simt_decode_bytelz(entry, fmt, comps, caps, byte_order=A.ENDIAN_DEFAULT, lz4_verify=0, flag_lz=False, lzss=None, size_only=0):
    """One emulated warp (byte-LZ kernel) or parser / resolver warp pair (flag_lz: the flag-LZ kernel) decodes `comps`."""
    n = len(comps)
    off, pos = [], 7
    for c in comps:
        off.append(pos)
        pos += len(c) + (pos % 5)
    limit = (pos + 15) & ~15
    backing = np.zeros(limit + 64, dtype=np.uint8)
    a0 = (-backing.ctypes.data) % 16
    src = backing[a0:a0 + limit]
    for o, c in zip(off, comps):
        src[o:o + len(c)] = np.frombuffer(c, dtype=np.uint8)
    doff, dpos = [], 0
    for i, c in enumerate(caps):
        doff.append(dpos)
        dpos += ((c + 8 + 15) & ~15) + (16 if i % 2 else 3)   # aligned and unaligned destinations
    dst = np.full(dpos + 8, 0xEE, dtype=np.uint8)
    out_len, consumed = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint64)
    status = np.full(n, 77, dtype=np.int32)
    u64 = lambda v: np.asarray(v, dtype=np.uint64)
    src_off, src_len, dst_off, dst_cap = u64(off), u64([len(c) for c in comps]), u64(doff), u64(caps)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    if flag_lz:
        lz = lzss if lzss is not None else A.lz_props_bits(12, 4, 2)   # LZSS.DefaultProperties (api.cu fill_decode_params)
        head = (C.c_int(fmt), C.c_int(byte_order), C.c_int(0), (C.c_int * 6)(lz.windows_bits, lz.length_bits, lz.min_length, lz.max_distance, lz.windows_start, 0))
    else:
        head = (C.c_int(fmt), C.c_int(byte_order), C.c_int(lz4_verify), C.c_int(size_only))
    rc = entry(*head, p(src), C.c_uint64(limit), p(src_off), p(src_len), p(dst), p(dst_off), p(dst_cap), p(out_len), p(consumed), p(status),
               C.c_uint32(n))
    assert rc == 0
    outs = []
    for i in range(n):
        assert (dst[doff[i] + caps[i]:doff[i] + caps[i] + 8] == 0xEE).all(), f"stream {i}: bytes written past the capacity"
        outs.append(dst[doff[i]:doff[i] + min(int(out_len[i]), caps[i])].tobytes())
    return outs, out_len, consumed, status


@pytest.mark.parametrize("fmt", BYTE_FORMATS, ids=fmt_id)
def test_bytelz_decoder_on_emulated_lanes(simt_bytelz_dec, oracle, bmp, fmt):
    from tests.util import corrupt
    rng = np.random.default_rng(404 + fmt)
    raws = [bmp[:n] for n in (33, 4097, 9000, 70000)] + [synth(rng, int(n), i % 5) for i, n in enumerate([5, 6, 31, 32, 33, 64, 65, 1000, 4096, 6000, 12000, 70000])]
    streams, caps = [], []
    for q in (0, 8):
        comps, st = oracle.encode_batch(fmt, raws, A.make_opts(quality=q))
        for i, (c, r) in enumerate(zip(comps, raws)):
            if st[i] != 0:
                continue
            streams.append(c)
            caps.append(len(r))
            if len(r) <= 12000:
                for mode in range(5):   # truncated, one byte flipped, garbage appended, empty, cut inside the header
                    streams.append(corrupt(rng, c, mode))
                    caps.append(len(r) if i % 2 else len(r) + 100)
                streams.append(c)       # destination one byte short
                caps.append(max(len(r) - 1, 0))
    ref, rlen, rcons, rst = oracle.decode_batch(fmt, streams, caps, A.make_opts())
    got, out_len, consumed, status = simt_decode_bytelz(simt_bytelz_dec, fmt, streams, caps)
    bad = [(i, int(status[i]), int(rst[i]), int(out_len[i]), int(rlen[i]), int(consumed[i]), int(rcons[i])) for i in range(len(streams))
           if status[i] != rst[i] or out_len[i] != rlen[i] or consumed[i] != rcons[i]]
    assert not bad, f"{fmt_id(fmt)}: (stream, status, ref, out_len, ref, consumed, ref) {bad[:5]} of {len(bad)}"
    assert all(g == r for g, r, s in zip(got, ref, rst) if s == 0)
    assert (rst == 0).sum() >= len(raws)


# ---- the flag-LZ decode kernel (csrc/decode_flaglz.cu, the headline kernel): one stream slot = a parser warp and a resolver warp
#      (64 fibers) handing batches over through two emulated named barriers
@pytest.fixture(scope="session")
def simt_flaglz_dec():
    f = _build("decode_flaglz", "flaglz_dec_harness.cpp", "DEC_DEVICE_INC").simt_decode_flaglz
    f.restype = C.c_int
    return f


FLAG_DEC_FORMATS = [A.FMT_LZ10, A.FMT_LZ11, A.FMT_YAZ0, A.FMT_YAZ1, A.FMT_LZSS, A.FMT_MIO0, A.FMT_YAY0, A.FMT_LZHUDSON, A.FMT_LZ40, A.FMT_LZ60,
                    A.FMT_SMSR00]


@pytest.mark.parametrize("fmt", FLAG_DEC_FORMATS, ids=fmt_id)
def test_flaglz_decoder_on_emulated_lanes(simt_flaglz_dec, oracle, bmp, fmt):
    from tests.util import corrupt
    rng = np.random.default_rng(808 + fmt)
    raws = [bmp[:n] for n in (33, 4097, 9000, 70000)] + [synth(rng, int(n), i % 5) for i, n in enumerate([1, 6, 31, 32, 33, 64, 65, 1000, 4096, 6000, 12000, 70000])]
    streams, caps = [], []
    for q in (0, 8):
        comps, st = oracle.encode_batch(fmt, raws, A.make_opts(quality=q))
        for i, (c, r) in enumerate(zip(comps, raws)):
            if st[i] != 0:
                continue
            streams.append(c)
            caps.append(len(r))
            if len(r) <= 12000:
                for mode in range(5):   # truncated, one byte flipped, garbage appended, empty, cut inside the header
                    streams.append(corrupt(rng, c, mode))
                    caps.append(len(r) if i % 2 else len(r) + 100)
                streams.append(c)       # destination one byte short
                caps.append(max(len(r) - 1, 0))
    ref, rlen, rcons, rst = oracle.decode_batch(fmt, streams, caps, A.make_opts())
    got, out_len, consumed, status = simt_decode_bytelz(simt_flaglz_dec, fmt, streams, caps, flag_lz=True)
    bad = [(i, int(status[i]), int(rst[i]), int(out_len[i]), int(rlen[i]), int(consumed[i]), int(rcons[i])) for i in range(len(streams))
           if status[i] != rst[i] or out_len[i] != rlen[i] or consumed[i] != rcons[i]]
    assert not bad, f"{fmt_id(fmt)}: (stream, status, ref, out_len, ref, consumed, ref) {bad[:5]} of {len(bad)}"
    assert all(g == r for g, r, s in zip(got, ref, rst) if s == 0)
    assert (rst == 0).sum() >= len(raws)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_random_lane_order(simt_lib, simt_flaglz_dec, simt_bytelz_dec, oracle, bmp, seed, monkeypatch):
    """SIMT_SHUFFLE: the emulated lanes run in a new random order on every scheduler pass.  A lane that reads what another lane
    wrote earlier in program order without a warp primitive / barrier in between then sees stale data some of the time, so
    equality with the oracle under random orders is evidence that the kernels' intra-warp and parser / resolver orderings are
    all explicit."""
    monkeypatch.setenv("SIMT_SHUFFLE", str(seed))
    rng = np.random.default_rng(seed)
    raws = [bmp[:9000], synth(rng, 6000, 0), synth(rng, 6000, 1), synth(rng, 12000, 2), synth(rng, 5000, 3), synth(rng, 3000, 4), bmp[5000:5033]]
    for fmt, q in ((A.FMT_LZ10, 8), (A.FMT_YAY0, 10), (A.FMT_LZ11, 3)):
        _check(simt_lib, oracle, fmt, raws, q)
    for fmt in (A.FMT_LZ4, A.FMT_SNAPPY, A.FMT_LZO):
        _check(simt_lib, oracle, fmt, raws, 8, seq=True)
    for fmt, entry, flag in ((A.FMT_LZ10, simt_flaglz_dec, True), (A.FMT_YAZ0, simt_flaglz_dec, True), (A.FMT_MIO0, simt_flaglz_dec, True),
                             (A.FMT_LZ4_BLOCK, simt_bytelz_dec, False), (A.FMT_LZO, simt_bytelz_dec, False), (A.FMT_PRS, simt_bytelz_dec, False)):
        comps, st = oracle.encode_batch(fmt, raws, A.make_opts(quality=8))
        caps = [len(r) for r in raws]
        ref, rlen, rcons, rst = oracle.decode_batch(fmt, comps, caps, A.make_opts())
        got, out_len, consumed, status = simt_decode_bytelz(entry, fmt, comps, caps, flag_lz=flag)
        assert (status == rst).all() and (out_len == rlen).all() and (consumed == rcons).all(), fmt_id(fmt)
        assert all(g == r for g, r, s in zip(got, ref, rst) if s == 0), fmt_id(fmt)


def test_far_reference_right_after_a_drain_step(simt_bytelz_dec, oracle):
    """The stream on which tools/fuzz_simt_decode.py caught the byte-LZ decoder reading drained bytes back from global memory
    without a warp barrier after the drain step (422 of 4096 bytes stale on the emulation; lock-step execution hid it on the GPU)."""
    s = open(os.path.join(ROOT, "tests", "golden", "lzo_far_reference_after_drain.lzo"), "rb").read()
    ref, rlen, rcons, rst = oracle.decode_batch(A.FMT_LZO, [s], [4096], A.make_opts())
    got, out_len, consumed, status = simt_decode_bytelz(simt_bytelz_dec, A.FMT_LZO, [s], [4096])
    assert rst[0] == 0 and status[0] == 0 and out_len[0] == rlen[0] == 4096 and consumed[0] == rcons[0]
    assert got[0] == ref[0]


@pytest.mark.parametrize("fmt", BYTE_FORMATS, ids=fmt_id)
def test_bytelz_size_scan_on_emulated_lanes(simt_bytelz_dec, oracle, bmp, fmt):
    """size_only (aurora_decoded_size_batch's scan for the formats whose header does not carry the size): the same walk with the
    stores dropped — the decoded length of every valid stream, nothing written."""
    rng = np.random.default_rng(55 + fmt)
    raws = [bmp[:9000]] + [synth(rng, int(n), i % 5) for i, n in enumerate([5, 33, 1000, 4096, 6000, 12000, 70000])]
    comps, st = oracle.encode_batch(fmt, raws, A.make_opts(quality=8))
    keep = [i for i in range(len(raws)) if st[i] == 0]
    comps, raws = [comps[i] for i in keep], [raws[i] for i in keep]
    got, out_len, consumed, status = simt_decode_bytelz(simt_bytelz_dec, fmt, comps, [0] * len(comps), size_only=1)
    # (the kernel reports the length with DST_TOO_SMALL against the zero capacity; api.cu's size path reads out_len)
    assert (status == A.DST_TOO_SMALL).all() and [int(x) for x in out_len] == [len(r) for r in raws]
    assert [int(x) for x in consumed] == [len(c) for c in comps]


# ---- the IsMatch and GetDecompressedSize rules of csrc/ismatch.cu: the library runs them on the host for the magic formats and
#      in the IsMatch / offset-scan kernels for every format, so one CPU build of them checks both
@pytest.fixture(scope="session")
def simt_rules():
    lib = _build("ismatch", "ismatch_harness.cpp", "ISMATCH_DEVICE_INC")
    lib.simt_is_match_one.restype = C.c_int
    lib.simt_is_match_one.argtypes = [C.c_void_p, C.c_uint64, C.c_int]
    lib.simt_core_decoded_size.restype = C.c_int
    lib.simt_core_decoded_size.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    return lib


@pytest.mark.parametrize("fmt", MATCHABLE, ids=fmt_id)
def test_is_match_rules_on_the_cpu(simt_rules, oracle, bmp, fmt):
    blobs = is_match_blobs(oracle, bmp, fmt)
    got = [simt_rules.simt_is_match_one(b, len(b), fmt) for b in blobs]
    ref = [int(oracle.is_match(fmt, b)) for b in blobs]
    bad = [i for i in range(len(blobs)) if got[i] != ref[i]]
    assert not bad, f"{fmt_id(fmt)}: {len(bad)} of {len(blobs)} differ, first #{bad[0]} rule={got[bad[0]]} ref={ref[bad[0]]} blob={blobs[bad[0]][:24].hex()}"
    assert sum(got) > 0
    # every offset of a ROM-like image: the stream at offset i runs to the end of the image, as in the offset-scan kernel
    rng = np.random.default_rng(77 + fmt)
    image, _ = rom_like_image(oracle, rng, fmt, [bmp[1000:9000], bytes(3000), synth(rng, 5000, 0), synth(rng, 2500, 2)])
    a = np.frombuffer(image, dtype=np.uint8)
    got = [simt_rules.simt_is_match_one(a.ctypes.data + i, len(image) - i, fmt) for i in range(len(image))]
    ref = [int(oracle.is_match(fmt, image[i:])) for i in range(len(image))]
    bad = [i for i in range(len(image)) if got[i] != ref[i]]
    assert not bad, f"{fmt_id(fmt)}: {len(bad)} of {len(image)} offsets differ, first {bad[0]}"


def test_formats_without_an_is_match_rule(simt_rules):
    blob = bytes(range(64))
    for fmt in (A.FMT_LZ4_BLOCK, A.FMT_SNAPPY_BLOCK, A.FMT_GCLZ):
        assert simt_rules.simt_is_match_one(blob, len(blob), fmt) == -1, fmt_id(fmt)


@pytest.mark.parametrize("fmt", SIZED_FORMATS, ids=fmt_id)
def test_decoded_size_rules_on_the_cpu(simt_rules, oracle, fmt):
    blobs = decoded_size_blobs(oracle, fmt)
    for order in (A.ENDIAN_DEFAULT, A.ENDIAN_LITTLE, A.ENDIAN_BIG):
        opts = A.make_opts(byte_order=order)
        for b in blobs:
            size = C.c_uint64(77)
            st = simt_rules.simt_core_decoded_size(fmt, order, b, len(b), C.byref(size))
            rs, rst = oracle.decoded_size(fmt, b, opts)
            assert (size.value, st) == (rs, rst) or (st != 0 and rst != 0), (fmt_id(fmt), order, b[:16].hex(), size.value, st, rs, rst)
