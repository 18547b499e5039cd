"""The fixed-token G32 core of the flag-LZ decoder (LZ10, LZSS) on the CPU lane emulation, on streams built to hit the edges of
its match pass: a warp iteration (32 flag groups) queues its matches in a token pass and then decodes them one match per lane,
in rounds of 32.  Hand-made LZ10 streams give iterations with exactly 0, 1, 32, 33, 96 and 97 matches (97: the iteration is
cut at the group that passes the 96-entry queue budget) and groups whose 8 tokens are all matches; LZSS streams are encoded
with LzProperties other than the default, whose match tokens carry the length in another field and a window-relative offset.
Every stream is compared with the oracle, also with the lanes in random order."""
import ctypes as C

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests.test_simt_kernels import _build, simt_decode_bytelz
from tests.util import synth


@pytest.fixture(scope="module")
def flaglz_dec():
    f = _build("decode_flaglz", "flaglz_dec_harness.cpp", "DEC_DEVICE_INC").simt_decode_flaglz
    f.restype = C.c_int
    return f


def lz10_stream(rng, iterations, tail_groups=5):
    """An LZ10 stream of 32-group blocks; `iterations` lists, per block, the slots (0..255) that hold a match token.  A tail of
    a few groups leaves the last block to the token-by-token cut at the end of the input."""
    body, n = bytearray(), 0

    def group(match_slots):
        nonlocal n
        flag, toks = 0, bytearray()
        for j in range(8):
            if j in match_slots and n > 0:
                flag |= 0x80 >> j
                ln, d = int(rng.integers(3, 19)), int(rng.integers(1, min(n, 4096) + 1))
                toks += bytes([((ln - 3) << 4) | ((d - 1) >> 8), (d - 1) & 0xFF])
                n += ln
            else:
                toks.append(int(rng.integers(0, 256)))
                n += 1
        body.append(flag)
        body.extend(toks)

    for slots in iterations:
        slots = set(int(s) for s in slots)
        for g in range(32):
            group({s - 8 * g for s in slots if 8 * g <= s < 8 * g + 8})
    for g in range(tail_groups):
        group({int(rng.integers(0, 8))})
    return bytes([0x10]) + n.to_bytes(3, "little") + bytes(body), n


def _compare(oracle, dec, fmt, streams, caps, opts, lzss=None):
    ref, rlen, rcons, rst = oracle.decode_batch(fmt, streams, caps, opts)
    got, out_len, consumed, status = simt_decode_bytelz(dec, fmt, streams, caps, flag_lz=True, lzss=lzss)
    assert (rst == 0).all()
    assert (status == rst).all() and (out_len == rlen).all() and (consumed == rcons).all()
    assert all(g == r for g, r in zip(got, ref))


@pytest.mark.parametrize("shuffle", [None, 11])
def test_lz10_iterations_with_given_match_counts(flaglz_dec, oracle, shuffle, monkeypatch):
    if shuffle is not None:
        monkeypatch.setenv("SIMT_SHUFFLE", str(shuffle))
    rng = np.random.default_rng(2024)
    lit = []                                              # all-literal block first: every match has bytes behind it
    every_slot = [s for g in range(0, 32, 3) for s in range(8 * g, 8 * g + 8)]   # 11 groups with a match in every slot
    cases = []
    for counts in ([0, 1, 32, 33, 96], [96, 96, 1, 0, 97], [33, 32, 97, 96]):
        cases.append([lit] + [rng.choice(256, size=c, replace=False) for c in counts])
    cases.append([lit, every_slot, list(range(96)), list(range(160, 256)), list(range(256))])   # 96 in a row, 256: cut at 12 groups
    cases.append([lit, [8 * g + 7 for g in range(32)], [8 * g for g in range(32)], [255], [0]])    # one match per group
    streams, caps = [], []
    for blocks in cases:
        s, n = lz10_stream(rng, blocks)
        streams.append(s)
        caps.append(n)
    _compare(oracle, flaglz_dec, A.FMT_LZ10, streams, caps, A.make_opts())


@pytest.mark.parametrize("props", [(10, 6, 2), (11, 5, 1), (8, 8, 2), ("w", 0x1000, 18, 3, 0xFEE)], ids=str)
def test_lzss_other_properties(flaglz_dec, oracle, bmp, props):
    lz = A.lz_props_window(*props[1:]) if props[0] == "w" else A.lz_props_bits(*props)
    rng = np.random.default_rng(77)
    raws = [bmp[:20000], bmp[30000:37000]] + [synth(rng, 9000, k) for k in range(5)]
    opts = A.make_opts(lzss=lz, quality=8)
    comps, st = oracle.encode_batch(A.FMT_LZSS, raws, opts)
    assert (st == 0).all()
    _compare(oracle, flaglz_dec, A.FMT_LZSS, comps, [len(r) for r in raws], opts, lzss=lz)
