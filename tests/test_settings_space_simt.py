"""The option values the other encoder and decoder tests leave at their defaults, on the CPU lane emulation (tests/simt):

  * CompressionSettings.MaxWindowBits, which widens every format's window and chain table (api.cu fill_encode_params) and so
    sends the flag formats to the sequential replay and writes distances the formats' tokens cannot hold (the reference's
    token writers truncate them; the oracle's bytes stay the contract);
  * the LZSS properties the decoder accepts (windows_bits 1-12, length_bits 1-8, max_distance 2-4096, min_length 1-255): small
    rings with a negative windows_start, one-byte matches, non-power-of-two windows, and flag groups longer than the g32 cores
    of decode_flaglz.cu take, which run the token-per-lane core.

The same sets run on the GPU in tests/test_settings_space_gpu.py."""
import ctypes as C

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests import tokens as T
from tests.test_simt_kernels import BYTE_FORMATS, PAR_FORMATS, SimtLibs, _build, _check, finder_params, simt_decode_bytelz
from tests.util import corrupt, fmt_id, synth

MWB = [0, 7, 12, 13, 16, 17, 20, 28]
# in tests/tokens.py's notation: (windows_bits, length_bits, threshold) for lz_props_bits, ("w", size, max_length, min_length,
# windows_start) for lz_props_window
LZSS_SETS = [(12, 8, 32), (12, 8, 33), ("w", 0x1000, 288, 33, 0), ("w", 0x1000, 289, 34, 0),   # the g32 / token-per-lane boundaries
             (12, 8, 40), (12, 8, 254), (12, 1, 254),                                          # long groups, long tokens
             (12, 4, 0),                                                                       # one-byte matches
             (7, 8, 2), (4, 4, 2), (2, 2, 1), (1, 3, 0),                                       # rings of 128 bytes down to 2
             ("w", 3000, 18, 3, 0), ("w", 1000, 66, 3, 0x3BE)]                                 # non-power-of-two windows
FILLS = [0, 0x20, 0xFF]
G32_GROUP_BYTES = 2304   # decode_flaglz.cu: the largest flag group (8 tokens) the g32 cores take


def lzss_id(p):
    return f"win({p[1]},{p[2]},{p[3]},{p[4]:#x})" if p[0] == "w" else f"bits({p[0]},{p[1]},{p[2]})"


def group_bytes(lz):
    """the most output bytes one flag group of 8 tokens can produce"""
    return 8 * ((1 << lz.length_bits) - 1 + lz.min_length)


def far_repeats(rng, bmp, block, gaps):
    """a noise block repeated after stretches of bitmap bytes: each copy lies block + gap bytes behind the next, so which copies
    a finder reaches depends on its window"""
    blk = rng.integers(0, 256, size=block, dtype=np.uint8).tobytes()
    out, pos = blk, 0
    for g in gaps:
        out += bmp[pos:pos + g] + blk
        pos += g + 50000
    return out


def par_supported(fmt, quality, lzss=None, max_window_bits=0):
    """encode_lz_par.cu encode_lz_par_supported: whether the lane-per-position search takes these settings (otherwise the
    device runs the sequential replay, whichever finder is asked for)"""
    if fmt in BYTE_FORMATS:
        return False
    f, _ = finder_params(fmt, quality, lzss=lzss, max_window_bits=max_window_bits)
    max_chain, lazy, hash_bits, chain_bits, min_len, max_len, min_dist, max_dist = f[:8]
    lz11 = fmt in (A.FMT_LZ11, A.FMT_LZ40, A.FMT_LZ60)
    return (lz11 or max_len <= 288) and max_dist <= 4096 and chain_bits >= 12 and min_len >= 1 and min_dist >= 1 and \
        not (f[9] and min_len == 1)


def lzss_raws(rng, bmp):
    return [bmp[:9000], synth(rng, 6000, 0), synth(rng, 5000, 1), synth(rng, 4000, 3), bytes(3000), b"ab" * 1500, bmp[:40]]


def lzss_token_streams(p, seed, per_profile):
    """grammar-built LZSS streams of one property set: `per_profile` from each of tests/tokens.py's profiles"""
    rng = np.random.default_rng(seed)
    return [T.generate(A.FMT_LZSS, rng, prof, size=int(rng.choice([300, 2000, 6000])), lzss_props=p)
            for prof in T.profiles_of(A.FMT_LZSS) for _ in range(per_profile)]


def lzss_decode_cases(oracle, p, seed, per_profile=2):
    """-> (streams, capacities): token streams, and the oracle's encodes valid, truncated, bit-flipped and one byte short"""
    lz = T.lzss_props(p)
    rng = np.random.default_rng(seed)
    streams, caps = [], []
    for s in lzss_token_streams(p, seed, per_profile):
        streams.append(s.data)
        caps.append(T.out_len([it for b in s.program for it in b]))
    raws = lzss_raws(rng, bytes(rng.integers(0, 256, size=9000, dtype=np.uint8)))
    comps, st = oracle.encode_batch(A.FMT_LZSS, raws, A.make_opts(quality=8, lzss=lz))
    assert (st == 0).all()
    for c, r in zip(comps, raws):
        streams += [c, corrupt(rng, c, 0), corrupt(rng, c, 1), c]
        caps += [len(r), len(r) + 100, len(r), max(len(r) - 1, 0)]
    return streams, caps


def test_the_sets_reach_both_decode_cores():
    """At least one set's flag group is longer than the g32 cores take (the token-per-lane core decodes it) and one is exactly
    as long: a later edit of LZSS_SETS cannot drop the token-per-lane core again without this failing."""
    sizes = [group_bytes(T.lzss_props(p)) for p in LZSS_SETS]
    assert any(s > G32_GROUP_BYTES for s in sizes) and G32_GROUP_BYTES in sizes


@pytest.fixture(scope="module")
def simt_lib():
    return SimtLibs()


@pytest.fixture(scope="module")
def simt_flaglz_dec():
    f = _build("decode_flaglz", "flaglz_dec_harness.cpp", "DEC_DEVICE_INC").simt_decode_flaglz
    f.restype = C.c_int
    return f


@pytest.mark.parametrize("fmt", PAR_FORMATS + BYTE_FORMATS, ids=fmt_id)
def test_max_window_bits_on_both_finders(simt_lib, oracle, bmp, fmt):
    """Every MaxWindowBits value, at qualities 1 and 8: bytes equal to the oracle's, on both emulated finders where the
    lane-per-position search takes the settings (up to 12 bits; the byte formats have the sequential replay only).  The inputs repeat a block at 6 500, 9 500 and 67 500 bytes: windows of 12, 13, 16 and
    17 bits each reach a different set of the copies."""
    rng = np.random.default_rng(700 + fmt)
    far = far_repeats(rng, bmp, 1500, [5000, 8000, 66000])
    raws = [far, bmp[:5000], synth(rng, 3000, 1), synth(rng, 2000, 2)]
    for mwb in MWB:
        for q in (1, 8):
            for seq in ((False, True) if par_supported(fmt, q, max_window_bits=mwb) else (True,)):
                _check(simt_lib, oracle, fmt, raws, q, seq=seq, skew=mwb % 16, max_window_bits=mwb)


def test_chain_slots_that_alias(simt_lib, oracle, bmp):
    """A stream longer than the chain table: at quality 1 and MaxWindowBits 28 the table has 2^18 slots, and a 300 KiB stream
    reuses them.  (Only MaxWindowBits makes a chain table this large for a format whose window is 4 KiB.)"""
    raw = bmp[:300 * 1024]
    _check(simt_lib, oracle, A.FMT_LZ10, [raw], 1, seq=True, max_window_bits=28)


@pytest.mark.parametrize("p", LZSS_SETS, ids=lzss_id)
def test_lzss_properties_encode(simt_lib, oracle, bmp, p):
    lz = T.lzss_props(p)
    rng = np.random.default_rng(900 + LZSS_SETS.index(p))
    raws = lzss_raws(rng, bmp)
    caps = [3 * len(r) + 256 for r in raws]   # (a two-byte token per one-byte match: output up to twice the input and the flags)
    for q in (0, 8, 10):
        for seq in ((False, True) if par_supported(A.FMT_LZSS, q, lzss=lz) else (True,)):
            _check(simt_lib, oracle, A.FMT_LZSS, raws, q, seq=seq, skew=q + seq, lzss=lz, caps=caps)


@pytest.mark.parametrize("p", LZSS_SETS, ids=lzss_id)
def test_lzss_properties_decode(simt_flaglz_dec, oracle, p):
    """Grammar-built and oracle-encoded streams of each set under each initial fill: status, out_len, consumed and bytes equal
    to the oracle's.  (Some sets do not round-trip in the reference itself: the u16 token drops offset bits.  The contract is
    the oracle's answer, so none is asserted.)"""
    lz = T.lzss_props(p)
    streams, caps = lzss_decode_cases(oracle, p, 1100 + LZSS_SETS.index(p), per_profile=1)
    for fill in FILLS:
        opts = A.make_opts(lzss=lz, lzss_initial_fill=fill)
        ref, rlen, rcons, rst = oracle.decode_batch(A.FMT_LZSS, streams, caps, opts)
        got, out_len, consumed, status = simt_decode_bytelz(simt_flaglz_dec, A.FMT_LZSS, streams, caps, flag_lz=True, lzss=lz,
                                                            initial_fill=fill)
        bad = [(i, int(status[i]), int(rst[i]), int(out_len[i]), int(rlen[i]), int(consumed[i]), int(rcons[i])) for i in range(len(streams))
               if status[i] != rst[i] or out_len[i] != rlen[i] or consumed[i] != rcons[i] or (rst[i] == 0 and got[i] != ref[i])]
        assert not bad, f"{lzss_id(p)} fill {fill:#x}: (stream, status, ref, out_len, ref, consumed, ref) {bad[:5]} of {len(bad)}"
        assert (rst == 0).sum() >= len(streams) // 4
