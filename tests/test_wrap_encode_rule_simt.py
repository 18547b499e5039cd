"""The wrapper encode rules as the library runs them on the host (aurora_encode_batch) and on the device (the plan and finish
kernels of aurora_encode_batch_device): wrap_encode_opts, wrap_encode_plan, wrap_encode_piece, wrap_encode_finish and the
ChunkLZ10 compaction / header writers in csrc/wrappers.cu, compiled for the CPU from the real file (everything above its
"// ---- kernel" line).  Every core piece the plan names is encoded by the oracle's core encoder and placed where the plan
says; the finish rule's copies, moves and header bytes then have to give the oracle's wrapped stream byte for byte.  Statuses
and out_len follow aurora_encode_batch's rules, pinned where the reference has no notion of them (a destination that is
too small for a core piece reports DST_TOO_SMALL with out_len 0).  No GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests.test_wrappers import _opt_sets
from tests.util import fmt_id, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIMT = os.path.join(ROOT, "tests", "simt")
CSRC = os.path.join(ROOT, "auroralib", "compression_b200", "csrc")
MAX_PIECES = 1 << 16
LENGTHS = [0, 1, 16, 17, 100, 4096, 4097, 20000, 70000]
SENTINEL = 0xEE
LEVEL5_EMPTY = bytes([1, 0, 0, 0])   # Level5 (type 1) of an empty input: the type word and no body
# the LZSS-property family: header bytes in front of the body, and whether the body uses LZSS.Lzss0Properties
FAMILY = {A.FMT_AKLZ: (16, False), A.FMT_LZ01: (16, True), A.FMT_FCMP: (12, True), A.FMT_IECP: (8, True), A.FMT_MDB4: (32, False),
          A.FMT_LZSEGA: (8, False), A.FMT_GCZ: (4, True), A.FMT_LZ00: (64, True)}


@pytest.fixture(scope="module")
def enc_rule(tmp_path_factory):
    build = tmp_path_factory.mktemp("wrap_encode_rule")
    src = open(os.path.join(CSRC, "wrappers.cu")).read()
    inc = build / "wrappers_device.inc"
    inc.write_text(src[:src.index("// ---- kernel\n")])
    so = build / "libsimt_wrap_encode_rule.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", SIMT, "-I", CSRC,
                           f'-DAURORA_REAL_COMMON="{os.path.join(CSRC, "common.cuh")}"', f'-DWRAPPERS_DEVICE_INC="{inc}"',
                           os.path.join(SIMT, "wrap_encode_rule_harness.cpp"), "-o", str(so)])
    lib = C.CDLL(str(so))
    lib.simt_wrap_encode_plan.restype = C.c_int64
    lib.simt_wrap_encode_plan.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.simt_wrap_encode_finish.restype = None
    lib.simt_wrap_encode_finish.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_char_p,
                                            C.c_void_p, C.c_void_p]
    return lib


def core_props(fmt):
    """the LzProperties the format fixes for its LZSS core (None: not an LZSS core)"""
    lzss0 = A.lz_props_window(0x1000, 0xF + 3, 3, 0xFEE, 1)
    if fmt == A.FMT_LEVEL5_LZSS:
        return lzss0
    if fmt == A.FMT_ECD:
        return A.lz_props_window(0x400, 0x42, 3, 0x3BE, 1)
    if fmt in FAMILY:
        return lzss0 if FAMILY[fmt][1] else A.lz_props_bits(12, 4, 2)
    return None


def lz00_keystream(body, key):
    """LZ00.cs:112-139: every byte XORed with a value of the LCG key, stepped before each byte"""
    out = bytearray(body)
    k = key
    for i in range(len(out)):
        k = (k * 1103515245 + 12345) & 0xFFFFFFFF
        t = (k >> 16) & 0x7FFF
        out[i] ^= (((t << 8) - t) >> 15) & 0xFF
    return bytes(out)


def stored_ecd(raw):
    n = len(raw).to_bytes(4, "big")
    return b"ECD\x00" + bytes(4) + n + n + raw


class Rule:
    """plan -> oracle core pieces -> finish for one (format, options, raw) at any capacity; core outputs are cached per piece"""

    def __init__(self, lib, oracle, fmt, kw, raw):
        self.lib, self.oracle, self.fmt, self.raw = lib, oracle, fmt, raw
        self.kw = {"quality": 8} | kw
        self.opts = A.make_opts(**self.kw)
        props = core_props(fmt)
        self.core_opts = A.make_opts(**self.kw, lzss=props) if props is not None else self.opts
        self.cache = {}

    def plan(self, cap):
        info = np.zeros(6, dtype=np.int64)
        pieces = np.zeros(4 * MAX_PIECES, dtype=np.uint64)
        k = self.lib.simt_wrap_encode_plan(self.fmt, C.addressof(self.opts), len(self.raw), cap, info.ctypes.data, pieces.ctypes.data,
                                           MAX_PIECES)
        assert k >= 0
        return [int(x) for x in info], pieces[:4 * k].reshape(k, 4).tolist()

    def core(self, core, soff, slen):
        key = (core, soff, slen)
        if key not in self.cache:
            c, st = self.oracle.encode(core, self.raw[soff:soff + slen], self.core_opts)
            assert st == A.OK, (fmt_id(self.fmt), core, slen)
            if self.fmt == A.FMT_LZ00:   # the body goes under the keystream
                c = c[:16] + lz00_keystream(c[16:], self.opts.lz00_key)
            self.cache[key] = c
        return self.cache[key]

    def run(self, cap):
        """-> (status, out_len, window bytes [0, out_len)), with the plan's info; nothing written past cap"""
        info, pieces = self.plan(cap)
        status, stored, chunked, npieces, core, head = info
        d = np.full(cap + 64, SENTINEL, dtype=np.uint8)
        r_out = np.zeros(max(1, npieces), dtype=np.uint64)
        r_st = np.zeros(max(1, npieces), dtype=np.int32)
        for k, (soff, slen, doff, dcap) in enumerate(pieces):
            assert doff + dcap <= cap, (fmt_id(self.fmt), cap, k)
            c = self.core(core, soff, slen)
            r_out[k] = len(c)
            r_st[k] = A.OK if len(c) <= dcap else A.DST_TOO_SMALL   # the encoder's bytes up to its capacity, then the needed size
            w = np.frombuffer(c[:dcap], dtype=np.uint8)
            d[doff:doff + len(w)] = w
        out = np.zeros(2, dtype=np.int64)
        self.lib.simt_wrap_encode_finish(self.fmt, C.addressof(self.opts), len(self.raw), cap, r_out.ctypes.data, r_st.ctypes.data,
                                         self.raw, d.ctypes.data, out.ctypes.data)
        assert (d[cap:] == SENTINEL).all(), (fmt_id(self.fmt), cap, "written past the capacity")
        out_len, st = int(out[0]), int(out[1])
        return st, out_len, d[:min(out_len, cap)].tobytes(), info


def host_answer(fmt, kw, raw, cap, ref, ref_st):
    """(status, out_len, bytes) that aurora_encode_batch gives, read from its rules, with the oracle's stream `ref`"""
    q = kw.get("quality", 8)
    n = len(raw)
    ok = lambda b: (A.OK, len(b), b)
    small = (A.DST_TOO_SMALL, 0, b"")
    if fmt == A.FMT_LZ77 and kw.get("lz77_type", 0x10) not in (0x10, 0x11, 0xF7):
        return A.NOT_SUPPORTED, 0, b""
    if fmt == A.FMT_LEVEL5 and q != 0 and kw.get("level5_type", 1) > 1:
        return A.NOT_SUPPORTED, 0, b""
    if fmt == A.FMT_LEVEL5 and q == 0:
        return ok(ref) if cap >= 4 + n else small
    if fmt == A.FMT_ECD:
        plain = kw.get("ecd_plain_size", 4) or 4
        if q == 0 or n <= 16:
            return ok(ref) if cap >= 16 + n else small
        if plain > n:
            return A.INVALID_ARGUMENT, 0, b""
        if cap < plain:
            return small
        if ref[3] == 1 and cap >= len(ref):
            return ok(ref)
        return ok(stored_ecd(raw)) if cap >= 16 + n else small   # the body does not shrink, or has no room: stored
    if fmt == A.FMT_LZ77 and kw.get("lz77_type") == 0xF7:
        chunk = kw.get("lz77_chunk_size", 0) or 0x1000
        if chunk < n:
            segs = (n + chunk - 1) // chunk
            if 8 + 2 * segs + segs * (chunk + chunk // 8 + 64) > cap:   # every chunk has a worst-case slot
                return small
            return ok(ref) if ref_st == A.OK else (ref_st, 0, b"")   # end offsets past 0xFFFF: INVALID_ARGUMENT
    assert ref_st == A.OK
    # the core piece must fit where the header leaves it room; the bytes the finish rule drops (Level5's LZ10 header, the
    # 16-byte LZSS header under a shorter family header) count
    extra = 0
    if fmt == A.FMT_LEVEL5:
        extra = 4 if n > 0xFFFFFF else 0
    elif fmt in FAMILY and FAMILY[fmt][0] < 16:
        extra = 16 - FAMILY[fmt][0]
    head = {A.FMT_LZ_3DS: 8, A.FMT_LZON: 16, A.FMT_SDPC: 8, A.FMT_LEVEL5: 0, A.FMT_LEVEL5_LZSS: 0}.get(fmt, 4)
    if fmt in FAMILY:
        head = max(0, FAMILY[fmt][0] - 16)
    if cap < head:
        return small
    return ok(ref) if cap >= len(ref) + extra else small


def opt_sets(fmt):
    extra = {A.FMT_ECD: [dict(ecd_plain_size=5000)], A.FMT_LZ77: [dict(lz77_type=0x28), dict(lz77_type=0xF7, lz77_chunk_size=0x10)],
             A.FMT_LEVEL5: [dict(level5_type=2)]}
    return _opt_sets(fmt) + extra.get(fmt, [])


def inputs(fmt):
    rng = np.random.default_rng(7300 + fmt)
    out = []
    for i, n in enumerate(LENGTHS):
        out.append(synth(rng, n, i % 4))   # compressible
        if n >= 16:
            out.append(rng.integers(0, 256, size=n, dtype=np.uint8).tobytes())   # incompressible
    return out


def capacities(ref_len, n):
    big = 2 * n + 1024 + 8 + 2 * (n + 2) + 70 * (n // 16 + 2)
    return sorted({c for c in (0, 1, 3, 4, 7, 8, 11, 12, 15, 16, 17, 31, 32, 47, 48, 63, 64, ref_len - 1, ref_len, ref_len + 12,
                               ref_len + 16, 16 + n - 1, 16 + n, big) if c >= 0})


@pytest.mark.parametrize("fmt", A.WRAPPER_FORMATS, ids=fmt_id)
def test_encode_rules_against_the_oracle(enc_rule, oracle, fmt):
    checked = ok = 0
    for kw in opt_sets(fmt):
        for raw in inputs(fmt):
            if fmt == A.FMT_LZ77 and kw.get("lz77_chunk_size") == 0x10 and len(raw) > 4097:
                continue   # (4 096 chunks of 16 bytes are enough)
            rule = Rule(enc_rule, oracle, fmt, kw, raw)
            unsupported = kw.get("lz77_type", 0x10) == 0x28 or kw.get("level5_type", 1) == 2   # (the oracle has no such encoder)
            if unsupported:
                ref, ref_st = b"", A.NOT_SUPPORTED
            elif fmt == A.FMT_LEVEL5 and not raw and kw.get("quality", 8) != 0:
                ref, ref_st = LEVEL5_EMPTY, A.OK   # (the oracle cannot encode an empty Level5 stream)
            else:
                ref, ref_st = oracle.encode(fmt, raw, rule.opts)
            for cap in capacities(len(ref), len(raw)):
                st, out_len, got, info = rule.run(cap)
                want = host_answer(fmt, kw, raw, cap, ref, ref_st)
                what = (fmt_id(fmt), kw, len(raw), cap, info)
                assert (st, out_len) == want[:2], what + (st, out_len, want[:2])
                if st == A.OK:
                    assert got == want[2], what
                    ok += 1
                checked += 1
    assert ok > 50 and checked > ok


def test_level5_empty_stream_has_a_four_byte_header(enc_rule, oracle):
    """An empty Level5 input: LZ10's header is 0x10 00 00 00 (size 0 fits its u24), so the finish rule drops 4 bytes, not 8:
    Level5.cs:127 writes the type word and CompressHeaderless writes nothing for no input."""
    rule = Rule(enc_rule, oracle, A.FMT_LEVEL5, {}, b"")
    assert rule.core(A.FMT_LZ10, 0, 0) == bytes([0x10, 0, 0, 0])
    assert rule.run(64)[:3] == (A.OK, 4, LEVEL5_EMPTY)


def test_chunklz10_pieces_overlap_earlier_slots_only(enc_rule, oracle, bmp):
    """Every ChunkLZ10 chunk moves down to behind the chunks in front of it: onto earlier slots, never into a later one."""
    raw = bmp[:40000]
    for chunk in (0x400, 0x1000):
        rule = Rule(enc_rule, oracle, A.FMT_LZ77, dict(lz77_type=0xF7, lz77_chunk_size=chunk), raw)
        ref, st = oracle.encode(A.FMT_LZ77, raw, rule.opts)
        cap = 3 * len(raw)
        info, pieces = rule.plan(cap)
        assert info[2] == 1 and info[3] == len(pieces) == (len(raw) + chunk - 1) // chunk
        end, body, overlaps = 0, 8 + 2 * len(pieces), 0
        for k, (soff, slen, doff, dcap) in enumerate(pieces):
            c = rule.core(A.FMT_LZ10, soff, slen)
            dst = body + end
            assert dst + len(c) <= doff + dcap and (k + 1 == len(pieces) or dst + len(c) <= pieces[k + 1][2])
            overlaps += k > 0 and dst < doff   # lands on an earlier chunk's slot
            end += len(c)
        assert overlaps == len(pieces) - 1
        assert rule.run(cap)[:3] == (A.OK, len(ref), ref)
