"""The decoders' device source on the CPU lane emulation (see tests/test_simt_kernels.py), on streams written from each format's
grammar by tests/tokens.py rather than by the reference encoder: distance-1 LZ10 runs, LZ11 / LZ40 / LZ60 tokens up to 65 808
bytes, LZO's M1 forms, Snappy's copy-4 and far copy-2, PRS's long copies with a length byte, MIO0 / Yay0 sections in any order,
with gaps or overlapping, and flag-LZ iterations at the parser's queue and hand-off limits.

Each generated program is first replayed in plain Python and decoded by the oracle, which must agree; that checks the writers.
Then each stream runs valid, cut at a token boundary, cut inside a token, and with a destination of exactly the decoded size,
one byte short, zero bytes and a few bytes more; the emulated kernels must equal the oracle in status, out_len, consumed and
bytes, and write nothing past the capacity.  A last test counts, per format, the edges the profiles produced."""
import ctypes as C
import functools
from collections import Counter

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests import tokens as T
from tests.test_simt_kernels import _build, simt_decode_blz, simt_decode_bytelz
from tests.util import fmt_id

PER_PROFILE = 40   # streams per (format, profile)


@pytest.fixture(scope="module")
def decoders():
    out = {}
    for key, name, harness, macro, sym in (("flag", "decode_flaglz", "flaglz_dec_harness.cpp", "DEC_DEVICE_INC", "simt_decode_flaglz"),
                                           ("byte", "decode_bytelz", "bytelz_dec_harness.cpp", "DEC_DEVICE_INC", "simt_decode_bytelz"),
                                           ("blz", "decode_blz", "blz_harness.cpp", "BLZ_DEVICE_INC", "simt_decode_blz")):
        f = getattr(_build(name, harness, macro), sym)
        f.restype = C.c_int
        out[key] = f
    return out


@functools.lru_cache(maxsize=None)
def streams(fmt, per_profile=PER_PROFILE, seed=0):
    from oracle import oracle as O
    rng = np.random.default_rng(7919 * fmt + seed)
    return [T.generate(fmt, rng, p, oracle=O) for p in T.profiles_of(fmt) for _ in range(per_profile)]


def options_key(s):
    return int(s.opts.byte_order), None if s.lzss is None else tuple(getattr(s.lzss, k) for k in ("windows_bits", "length_bits", "min_length", "max_distance", "windows_start")), s.fill


def variants(rng, s):
    """(stream bytes, capacity) of one generated stream: valid, cut at a token boundary, cut inside a token, and destinations of
    the exact size, one byte short, zero bytes and a few bytes more"""
    n = len(s.expect) if s.expect is not None else T.out_len([it for b in s.program for it in b])
    d = s.data
    out = [(d, n), (d, max(n - 1, 0)), (d, 0), (d, n + int(rng.integers(1, 70)))]
    inner = [m for m in s.marks if 0 < m < len(d)]
    if inner:
        m = inner[int(rng.integers(0, len(inner)))]
        out.append((d[:m], n))
        k = int(rng.integers(0, len(inner)))
        lo, hi = (inner[k - 1] if k else 0), inner[k]
        if hi - lo > 1:
            out.append((d[:int(rng.integers(lo + 1, hi))], n))
    if len(d) > 1:
        out.append((d[:int(rng.integers(1, len(d)))], n + 16))
    return out


def emulate(decoders, fmt, datas, caps, s0):
    """the emulated kernel of `fmt` under the decode options of stream s0"""
    if fmt == A.FMT_BLZ:
        return simt_decode_blz(decoders["blz"], datas, caps)
    if fmt in T.FLAG_FORMATS:
        return simt_decode_bytelz(decoders["flag"], fmt, datas, caps, byte_order=int(s0.opts.byte_order), flag_lz=True, lzss=s0.lzss,
                                  initial_fill=s0.fill)
    return simt_decode_bytelz(decoders["byte"], fmt, datas, caps, byte_order=int(s0.opts.byte_order))


def compare(decoders, oracle, fmt, cases, what):
    """cases: (stream, bytes, capacity); grouped by decode options, decoded by the oracle and by the emulation"""
    groups = {}
    for s, data, cap in cases:
        groups.setdefault(options_key(s), []).append((s, data, cap))
    checked = 0
    for key, group in groups.items():
        datas, caps = [g[1] for g in group], [g[2] for g in group]
        ref, rlen, rcons, rst = oracle.decode_batch(fmt, datas, caps, group[0][0].opts)
        got, out_len, consumed, status = emulate(decoders, fmt, datas, caps, group[0][0])
        bad = [i for i in range(len(datas)) if status[i] != rst[i] or out_len[i] != rlen[i] or consumed[i] != rcons[i]
               or (rst[i] == 0 and got[i] != ref[i])]
        if bad:
            i = bad[0]
            pytest.fail(f"{fmt_id(fmt)} {what} {key}: {len(bad)}/{len(datas)} differ; first: profile {group[i][0].profile}, "
                        f"{len(datas[i])} bytes, cap {caps[i]}: status {status[i]} / {rst[i]}, out_len {out_len[i]} / {rlen[i]}, "
                        f"consumed {consumed[i]} / {rcons[i]}, bytes equal {got[i] == ref[i]}")
        checked += len(datas)
    return checked


@pytest.mark.parametrize("fmt", T.ALL, ids=fmt_id)
def test_writers_against_the_oracle(oracle, fmt):
    """Every valid program decodes, on the oracle, to what `replay` says, and consumes the whole stream (MIO0, Yay0 and BLZ
    stop where their sections end); the programs meant to be rejected are."""
    ss = streams(fmt)
    ok = [s for s in ss if s.expect is not None]
    for key in {options_key(s) for s in ss}:
        grp = [s for s in ss if options_key(s) == key]
        out, olen, cons, st = oracle.decode_batch(fmt, [s.data for s in grp], [len(s.expect) if s.expect is not None else 1 << 20 for s in grp], grp[0].opts)
        for i, s in enumerate(grp):
            if s.expect is None:
                assert st[i] != 0, (fmt_id(fmt), s.profile)
                continue
            assert st[i] == 0 and out[i] == s.expect, (fmt_id(fmt), s.profile, int(st[i]), len(out[i]), len(s.expect))
            if fmt not in (A.FMT_MIO0, A.FMT_YAY0, A.FMT_BLZ):
                assert cons[i] == len(s.data), (fmt_id(fmt), s.profile, int(cons[i]), len(s.data))
    assert len(ok) >= len(ss) * 9 // 10


@pytest.mark.parametrize("fmt", T.ALL, ids=fmt_id)
def test_emulated_decoders_on_token_streams(decoders, oracle, fmt):
    rng = np.random.default_rng(31 + fmt)
    cases = [(s, d, cap) for s in streams(fmt) for d, cap in variants(rng, s)]
    assert compare(decoders, oracle, fmt, cases, "token streams") == len(cases)


@pytest.mark.parametrize("fmt", [A.FMT_LZ10, A.FMT_LZ11, A.FMT_YAY0, A.FMT_LZSS, A.FMT_LZO, A.FMT_SNAPPY_BLOCK, A.FMT_PRS, A.FMT_LZ4_BLOCK],
                         ids=fmt_id)
def test_token_streams_in_random_lane_order(decoders, oracle, fmt, monkeypatch):
    """SIMT_SHUFFLE (see test_simt_kernels.test_random_lane_order) on a subset of the streams"""
    monkeypatch.setenv("SIMT_SHUFFLE", str(fmt))
    rng = np.random.default_rng(5 + fmt)
    ss = streams(fmt)[::4]
    cases = [(s, s.data, len(s.expect) if s.expect is not None else 4096) for s in ss]
    cases += [(s, d, cap) for s in ss[::3] for d, cap in variants(rng, s)[1:]]
    compare(decoders, oracle, fmt, cases, "shuffled lanes")


# ---- what every profile must keep producing, per format
def required(fmt):
    flag = fmt in T.FLAG_FORMATS
    spec = T.SPEC.get(fmt, T.SPEC[A.FMT_LZ10])
    req = [f"period{d}" for d in range(max(1, spec.dmin), 5)] + ["dmax"]
    req += ["rejected"] if fmt == A.FMT_BLZ else ["past_start"]
    if flag or fmt == A.FMT_BLZ:
        req += ["ring_wrap", "total_at_drain_step", "len_max"]
    else:
        req += ["byte_ring_dist", "source_straddles_drain"]
    if flag:
        req += [f"iter{k}" for k in (T.HANDOFF_AT - 1, T.HANDOFF_AT, T.HANDOFF_AT + 1, T.ITER_MATCHES, T.ITER_MATCHES + 1)]
        req += ["span-1", "span+0", "span+1", "chain", "chain_broken", "overlap_pair"]
    if fmt in (A.FMT_LZ11, A.FMT_LZ40, A.FMT_LZ60):
        req += ["len_over_16k", "len_2048k"]
    req += {A.FMT_LZ11: ["lz11_2", "lz11_3", "lz11_4"], A.FMT_LZ40: ["lz40_d0"], A.FMT_LZ60: ["lz40_d0"],
            A.FMT_MIO0: ["layout_codes_lits", "layout_lits_codes", "layout_gaps", "layout_overlap", "lits_first"],
            A.FMT_YAZ0: ["yaz_order0x", "yaz_order0", "yaz_order1"], A.FMT_YAZ1: ["yaz_order0x", "yaz_order0", "yaz_order1"],
            A.FMT_SMSR00: ["smsr_pad1"],
            A.FMT_LZ4_BLOCK: ["lz4_lit_ext_edge", "lz4_match_ext_edge", "lz4_match_tail"],
            A.FMT_LZ4_LEGACY: ["lz4_lit_ext_edge", "lz4_match_ext_edge"], A.FMT_LZ4: ["lz4_lit_ext_edge", "lz4_stored_block"],
            A.FMT_LZO: ["lzo_m1", "lzo_m1_far", "lzo_m2", "lzo_m3", "lzo_m4", "lzo_first_byte_run"],
            A.FMT_SNAPPY_BLOCK: ["snappy_c1", "snappy_c2", "snappy_c4", "snappy_tag60", "snappy_tag61", "snappy_tag62", "snappy_tag63"],
            A.FMT_SNAPPY: ["snappy_c4", "snappy_tag63", "snappy_stored_chunk", "snappy_skip_chunk"],
            A.FMT_PRS: ["prs_short", "prs_long", "prs_long_byte", "prs_order0", "prs_order1"]}.get(fmt, [])
    if fmt == A.FMT_YAY0:
        req += ["layout_codes_lits", "layout_lits_codes", "layout_gaps", "layout_overlap", "lits_first"]
    return req


def coverage(fmt, ss):
    c = Counter()
    for s in ss:
        c += T.classify(fmt, [it for b in s.program for it in b], T.spec_of(fmt, s.lzss))
        c += s.forms
        c["rejected"] += s.expect is None
    return c


@pytest.mark.parametrize("fmt", T.ALL, ids=fmt_id)
def test_profiles_reach_their_edges(fmt):
    c = coverage(fmt, streams(fmt))
    req = required(fmt)
    print(f"{fmt_id(fmt)}: " + ", ".join(f"{k} {c[k]}" for k in req))
    missing = [k for k in req if c[k] < 1]
    assert not missing, f"{fmt_id(fmt)}: the generators no longer produce {missing}; counts {dict(c)}"
