"""The encoders' device source on the CPU lane emulation (tests/simt) against the oracle encoder, on inputs built against the
finders' tables (tests/enc_inputs.py): both finders, every flag-LZ format, the byte-LZ writers on the sequential replay, several
streams per batch at varying source skews (one warp carries its tables from stream to stream, as on the device), and every
capacity edge of the token writers."""
import functools

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests import enc_inputs as E
from tests.test_simt_kernels import BYTE_FORMATS, PAR_FORMATS, SimtLibs, _check, simt_encode
from tests.util import fmt_id

# qualities where a profile's parameter changes: max_chain (every quality), the lazy threshold 3 + q / 3, the small-match table
QUALITIES = [0, 1, 2, 5, 6, 8, 9, 10]


@pytest.fixture(scope="module")
def simt_lib():
    return SimtLibs()


@functools.lru_cache(maxsize=None)
def flag_pairs(fmt, quality):
    p = E.Params(fmt, quality)
    out = []
    for name, fn in E.FLAG_PROFILES.items():
        kw = {"park": quality in (0, 8)} if name == "distance" else {}   # (the parking pass needs 16 KiB streams: two qualities)
        out += [(name,) + pair for pair in fn(p, 100 * quality + fmt, **kw)]
    if fmt == A.FMT_BLZ:   # BLZ compresses the reversed input: reverse the designs back
        out = [(name, what, a[::-1], b[::-1]) for name, what, a, b in out]
    return out


@functools.lru_cache(maxsize=None)
def byte_pairs(fmt, quality):
    return [("bytes",) + pair for pair in E.profile_bytes(E.Params(fmt, quality), fmt)]


def _raws(pairs):
    return [x for _, _, a, b in pairs for x in (a, b)]


def _round_trip(oracle, fmt, raws, quality, **kw):
    ref, st = oracle.encode_batch(fmt, raws, A.make_opts(quality=quality, **kw))
    outs, out_len, consumed, dst = oracle.decode_batch(fmt, ref, [len(r) for r in raws], A.make_opts(**{k: v for k, v in kw.items() if k == "lzss"}))
    bad = [i for i in range(len(raws)) if st[i] == 0 and not (dst[i] == 0 and outs[i] == raws[i])]
    assert not bad, f"{fmt_id(fmt)} q{quality}: the oracle's stream #{bad[0]} does not decode to its input"
    return ref


@pytest.mark.parametrize("fmt", PAR_FORMATS, ids=fmt_id)
@pytest.mark.parametrize("quality", QUALITIES)
def test_flag_formats_on_finder_edges(simt_lib, oracle, fmt, quality):
    raws = _raws(flag_pairs(fmt, quality))
    if E.Params(fmt, quality).min_table:
        raws = [bytes(40)] + E.head_at_start() + [bytes(40)] + raws   # zeros in front of the stream: the byte before position 0
    _round_trip(oracle, fmt, raws, quality)
    for seq in (False, True):
        _check(simt_lib, oracle, fmt, raws, quality, seq=seq, skew=(quality + seq) % 16)


@pytest.mark.parametrize("fmt", [A.FMT_LZ10, A.FMT_YAZ0, A.FMT_LZ11], ids=fmt_id)
@pytest.mark.parametrize("quality", [1, 8])
def test_compatibility_mode_on_short_periods(simt_lib, oracle, fmt, quality):
    raws = _raws([("compat",) + pr for pr in E.profile_compat(E.Params(fmt, quality), fmt)])
    _round_trip(oracle, fmt, raws, quality, strategy=A.STRATEGY_COMPATIBILITY)
    for seq in (False, True):
        _check(simt_lib, oracle, fmt, raws, quality, seq=seq, skew=5, strategy=A.STRATEGY_COMPATIBILITY)


@pytest.mark.parametrize("props", [(10, 6, 2), (11, 5, 2), (8, 8, 2)], ids=["1024", "2048", "256"])
@pytest.mark.parametrize("quality", [0, 8])
def test_lzss_windows(simt_lib, oracle, props, quality):
    lz = A.lz_props_bits(*props)
    p = E.Params(A.FMT_LZSS, quality, lzss=lz)
    raws = _raws([("distance",) + pr for pr in E.profile_distance(p, 11, park=False)] +
                 [("lazy",) + pr for pr in E.profile_lazy(p, 12)])
    _round_trip(oracle, A.FMT_LZSS, raws, quality, lzss=lz)
    for seq in (False, True):
        _check(simt_lib, oracle, A.FMT_LZSS, raws, quality, seq=seq, skew=9, lzss=lz)


@pytest.mark.parametrize("fmt", BYTE_FORMATS, ids=fmt_id)
@pytest.mark.parametrize("quality", [0, 8])
def test_byte_writers_on_planted_matches(simt_lib, oracle, fmt, quality):
    raws = _raws(byte_pairs(fmt, quality)) + (E.long_literal_runs() if fmt in (A.FMT_SNAPPY, A.FMT_SNAPPY_BLOCK) else [])
    _round_trip(oracle, fmt, raws, quality)
    _check(simt_lib, oracle, fmt, raws, quality, seq=True, skew=quality + 3)


@pytest.mark.parametrize("fmt", [f for f in PAR_FORMATS if f != A.FMT_BLZ] + BYTE_FORMATS, ids=fmt_id)
def test_every_profile_decides_its_edge(oracle, fmt):
    """Per format and quality, each pair's two inputs give reference outputs of different lengths: the edge changes the parse.
    (BLZ searches its input backwards; the reversed designs run through its finder but are not aimed at it.)"""
    cases = [(q, byte_pairs(fmt, q)) for q in (0, 8)] if fmt in BYTE_FORMATS else [(q, flag_pairs(fmt, q)) for q in QUALITIES]
    for q, pairs in cases:
        ref, st = oracle.encode_batch(fmt, _raws(pairs), A.make_opts(quality=q))
        same = [pairs[i // 2][:2] for i in range(0, len(ref), 2) if len(ref[i]) == len(ref[i + 1])]
        assert not same, f"{fmt_id(fmt)} q{q}: these pairs do not change the reference's output length: {same}"
        profiles = {name for name, *_ in pairs}
        p = E.Params(fmt, q)
        expected = {"bytes"} if fmt in BYTE_FORMATS else set(E.FLAG_PROFILES) - (set() if p.min_table and p.min_dist >= 2 else {"small"})
        assert profiles == expected, (fmt_id(fmt), q, profiles, expected)


# ---- capacities: exactly the needed size, one byte less, 0, 1, inside the header, inside the MIO0 / Yay0 / SMSR00 section copy
def capacity_points(fmt, ref):
    need = len(ref)
    pts = {need, need - 1, 0, 1, 3, 7, 15, need // 2}
    if fmt in (A.FMT_MIO0, A.FMT_YAY0):
        comp_off, lit_off = int.from_bytes(ref[8:12], "big"), int.from_bytes(ref[12:16], "big")
        pts |= {comp_off - 1, comp_off + 1, (comp_off + lit_off) // 2, lit_off + 1}
    if fmt == A.FMT_SMSR00:
        lit_off = int.from_bytes(ref[12:16], "big")
        pts |= {lit_off - 1, lit_off + 1}
    return sorted(c for c in pts if 0 <= c <= need)


def capacity_inputs(fmt):
    p = E.Params(fmt, 8)
    pairs = E.profile_bytes(p, 1) if fmt in BYTE_FORMATS else E.profile_lazy(p, 1)
    return [pairs[0][1], bytes(300), pairs[-1][2]]


@pytest.mark.parametrize("fmt", [f for f in PAR_FORMATS if f != A.FMT_BLZ] + BYTE_FORMATS, ids=fmt_id)
def test_capacity_sweep(simt_lib, oracle, fmt):
    """BLZ's body is reversed and its footer added on the host: its capacities are swept on the GPU only."""
    seq = fmt in BYTE_FORMATS
    for raw in capacity_inputs(fmt):
        ref, st = oracle.encode_batch(fmt, [raw], A.make_opts(quality=8))
        assert st[0] == 0
        caps = capacity_points(fmt, ref[0])
        for s in ((False, True) if not seq else (True,)):
            got, status, out_len = simt_encode(simt_lib, fmt, [raw] * len(caps), 8, caps=caps, seq=s, skew=7)
            for c, g, stt, ol in zip(caps, got, status, out_len):
                if c == len(ref[0]):
                    assert stt == A.OK and g == ref[0], (fmt_id(fmt), c)
                else:
                    # (simt_encode checks that the 8 bytes behind every capacity are untouched)
                    assert stt == A.DST_TOO_SMALL and int(ol) == len(ref[0]), (fmt_id(fmt), s, c, int(stt), int(ol), len(ref[0]))
