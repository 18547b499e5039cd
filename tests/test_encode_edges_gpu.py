"""The encoders on the B200 against the oracle on the finder-edge inputs of tests/enc_inputs.py: the host entry point with sources
packed at 1-byte offsets (the lane-per-position search then stages skewed lines), each finder forced and CompatibilityMode; the
device entry point on sentinel-filled tensors; the capacity edges of every format through both entry points; and the worst-case
inputs at the capacity aurora_encode_bound gives."""
import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests import enc_inputs as E
from tests.test_encode_edges_simt import byte_pairs, capacity_points, flag_pairs
from tests.test_encode_gpu import ENC_FORMATS
from tests.test_simt_kernels import BYTE_FORMATS, PAR_FORMATS
from tests.util import fmt_id

pytestmark = pytest.mark.gpu

SENTINEL = 0xEE


def _pack_tight(raws):
    """Sources back to back (1-byte offsets, 3 spare bytes behind each): every source skew occurs."""
    off, pos = [], 1
    for r in raws:
        off.append(pos)
        pos += len(r) + 3
    base = np.zeros(pos + 16, dtype=np.uint8)
    for o, r in zip(off, raws):
        base[o:o + len(r)] = np.frombuffer(r, dtype=np.uint8)
    return base, np.asarray(off, dtype=np.uint64), np.asarray([len(r) for r in raws], dtype=np.uint64)


def host_encode(codec, fmt, raws, caps, opts):
    """aurora_encode_batch on tightly packed sources, destinations with 16 sentinel bytes behind every capacity."""
    base, off, ln = _pack_tight(raws)
    doff = np.zeros(len(raws), dtype=np.uint64)
    pos = 0
    for i, c in enumerate(caps):
        doff[i] = pos
        pos += c + 16
    dst = np.full(pos + 16, SENTINEL, dtype=np.uint8)
    out_len, status = codec.encode_packed(fmt, base, off, ln, dst, doff, np.asarray(caps, dtype=np.uint64), opts)
    for i, c in enumerate(caps):
        assert (dst[int(doff[i]) + c:int(doff[i]) + c + 16] == SENTINEL).all(), f"{fmt_id(fmt)} stream {i}: written past the capacity {c}"
    outs = [dst[int(doff[i]):int(doff[i]) + min(int(out_len[i]), caps[i])].tobytes() for i in range(len(raws))]
    return outs, status, out_len


def device_encode(codec, fmt, raws, caps, opts):
    """aurora_encode_batch_device: offsets multiples of 16, sentinel-filled destination; nothing outside the windows may change."""
    import torch
    dev = torch.device("cuda", 0)
    soff, pos = [], 0
    for r in raws:
        soff.append(pos)
        pos += (len(r) + 15) & ~15
    src = np.zeros(pos + 16, dtype=np.uint8)
    for o, r in zip(soff, raws):
        src[o:o + len(r)] = np.frombuffer(r, dtype=np.uint8)
    doff, pos = [], 0
    for c in caps:
        doff.append(pos)
        pos += ((c + 15) & ~15) + 32
    d_src = torch.from_numpy(src).to(dev)
    d_dst = torch.full((pos + 32,), SENTINEL, dtype=torch.uint8, device=dev)
    t64 = lambda v: torch.tensor(v, dtype=torch.int64, device=dev)
    d_out_len = torch.full((len(raws),), -1, dtype=torch.int64, device=dev)
    d_status = torch.full((len(raws),), 77, dtype=torch.int32, device=dev)
    codec.encode_device(fmt, d_src, t64(soff), t64([len(r) for r in raws]), d_dst, t64(doff), t64(caps), d_out_len, d_status, opts)
    torch.cuda.synchronize(dev)
    dst = d_dst.cpu().numpy()
    out_len, status = d_out_len.cpu().numpy(), d_status.cpu().numpy()
    inside = np.zeros(len(dst), dtype=bool)
    for o, c in zip(doff, caps):
        inside[o:o + c] = True
    assert (dst[~inside] == SENTINEL).all(), f"{fmt_id(fmt)}: bytes outside the destination windows changed"
    return [dst[o:o + min(int(l), c)].tobytes() for o, c, l in zip(doff, caps, out_len)], status, out_len


def _expect_oracle(oracle, fmt, raws, opts, got, status):
    ref, rst = oracle.encode_batch(fmt, raws, opts)
    assert (status == rst).all(), (fmt_id(fmt), [(i, int(status[i]), int(rst[i])) for i in range(len(raws)) if status[i] != rst[i]][:5])
    bad = [i for i in range(len(raws)) if rst[i] == 0 and got[i] != ref[i]]
    assert not bad, f"{fmt_id(fmt)}: stream #{bad[0]} (len {len(raws[bad[0]])}) differs from the oracle: {len(got[bad[0]])} vs {len(ref[bad[0]])} bytes"
    return ref


FINDERS = [0, A.STRATEGY_PARALLEL_FINDER, A.STRATEGY_SERIAL_FINDER]


@pytest.mark.parametrize("fmt", PAR_FORMATS, ids=fmt_id)
@pytest.mark.parametrize("quality", [0, 2, 6, 8, 10])
def test_finder_edges_through_the_host_entry_point(codec, oracle, fmt, quality):
    raws = [x for _, _, a, b in flag_pairs(fmt, quality) for x in (a, b)]
    if E.Params(fmt, quality).min_table:
        raws = [bytes(40)] + E.head_at_start() + [bytes(40)] + raws
    caps = [codec.encode_bound(fmt, len(r)) for r in raws]
    for finder in FINDERS:
        opts = A.make_opts(quality=quality, strategy=finder)
        got, st, _ = host_encode(codec, fmt, raws, caps, opts)
        _expect_oracle(oracle, fmt, raws, opts, got, st)
    compat = [x for _, a, b in E.profile_compat(E.Params(fmt, quality), fmt) for x in (a, b)]
    for finder in FINDERS:
        opts = A.make_opts(quality=quality, strategy=finder | A.STRATEGY_COMPATIBILITY)
        got, st, _ = host_encode(codec, fmt, compat, [codec.encode_bound(fmt, len(r)) for r in compat], opts)
        _expect_oracle(oracle, fmt, compat, opts, got, st)


@pytest.mark.parametrize("fmt", BYTE_FORMATS, ids=fmt_id)
@pytest.mark.parametrize("quality", [0, 8])
def test_byte_writer_edges_through_the_host_entry_point(codec, oracle, fmt, quality):
    raws = [x for _, _, a, b in byte_pairs(fmt, quality) for x in (a, b)] + E.long_literal_runs()
    opts = A.make_opts(quality=quality)
    got, st, _ = host_encode(codec, fmt, raws, [codec.encode_bound(fmt, len(r)) for r in raws], opts)
    _expect_oracle(oracle, fmt, raws, opts, got, st)


@pytest.mark.parametrize("fmt", [f for f in ENC_FORMATS if f != A.FMT_BLZ], ids=fmt_id)
def test_device_entry_point_equals_the_host_entry_point(codec, oracle, fmt):
    pairs = byte_pairs(fmt, 8) if fmt in BYTE_FORMATS else flag_pairs(fmt, 8)
    raws = [x for _, _, a, b in pairs for x in (a, b)]
    raws = sorted(raws, key=len)   # the longest stream last: the MIO0 / Yay0 / SMSR00 scratch is sized from the lengths read back
    caps = [codec.encode_bound(fmt, len(r)) for r in raws]
    opts = A.make_opts(quality=8)
    hgot, hst, hlen = host_encode(codec, fmt, raws, caps, opts)
    dgot, dst, dlen = device_encode(codec, fmt, raws, caps, opts)
    assert (hst == dst).all() and (hlen == dlen.astype(np.uint64)).all() and hgot == dgot, fmt_id(fmt)
    _expect_oracle(oracle, fmt, raws, opts, dgot, dst)


def test_device_entry_point_many_small_streams(codec, oracle):
    """A few thousand short edge streams: resident warps take many streams each through the work ticket."""
    small = [x for _, _, a, b in flag_pairs(A.FMT_LZ10, 2) for x in (a, b) if len(x) < 2000]
    raws = (small * (3000 // len(small) + 1))[:3000]
    caps = [codec.encode_bound(A.FMT_LZ10, len(r)) for r in raws]
    opts = A.make_opts(quality=2)
    got, st, _ = device_encode(codec, A.FMT_LZ10, raws, caps, opts)
    _expect_oracle(oracle, A.FMT_LZ10, raws, opts, got, st)


def test_device_entry_point_refuses_blz_without_a_launch(codec):
    from auroralib.compression_b200 import AuroraError
    before = codec.kernel_launches
    with pytest.raises(AuroraError, match="NOT_SUPPORTED"):
        device_encode(codec, A.FMT_BLZ, [bytes(100)], [200], A.make_opts(quality=8))
    assert codec.kernel_launches == before


@pytest.mark.parametrize("fmt", ENC_FORMATS, ids=fmt_id)
def test_capacity_sweep(codec, oracle, fmt):
    """At the needed size: OK and the oracle's bytes; below it: DST_TOO_SMALL with out_len = the needed size, nothing written
    behind the capacity (the bytes of a failed stream below its capacity are unspecified)."""
    p = E.Params(fmt, 8)
    pairs = E.profile_bytes(p, 1) if fmt in BYTE_FORMATS else E.profile_lazy(p, 1)
    opts = A.make_opts(quality=8)
    for raw in (pairs[0][1], bytes(300), pairs[-1][2]):
        ref, rst = oracle.encode_batch(fmt, [raw], opts)
        assert rst[0] == 0
        caps = capacity_points(fmt, ref[0])
        entries = [host_encode] if fmt == A.FMT_BLZ else [host_encode, device_encode]
        for entry in entries:
            got, st, out_len = entry(codec, fmt, [raw] * len(caps), caps, opts)
            for c, g, s, ol in zip(caps, got, st, out_len):
                if c == len(ref[0]):
                    assert s == A.OK and g == ref[0], (fmt_id(fmt), entry.__name__, c)
                else:
                    assert s == A.DST_TOO_SMALL and int(ol) == len(ref[0]), (fmt_id(fmt), entry.__name__, c, int(s), int(ol), len(ref[0]))


@pytest.mark.parametrize("fmt", ENC_FORMATS, ids=fmt_id)
def test_worst_cases_fit_the_bound(codec, oracle, fmt):
    cases = E.worst_cases(200000)
    raws = list(cases.values())
    for q in (0, 8, 15):
        opts = A.make_opts(quality=q)
        if q == 15 and fmt not in BYTE_FORMATS:
            opts = A.make_opts(quality=q, strategy=A.STRATEGY_PARALLEL_FINDER)
        got, st, out_len = host_encode(codec, fmt, raws, [codec.encode_bound(fmt, len(r)) for r in raws], opts)
        ref, rst = oracle.encode_batch(fmt, raws, opts)
        assert (rst == 0).all() and (st == A.OK).all(), (fmt_id(fmt), q, list(st))
        assert [int(x) for x in out_len] == [len(r) for r in ref], (fmt_id(fmt), q)
        assert got == ref, (fmt_id(fmt), q)
