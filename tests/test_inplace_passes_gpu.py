"""GPU tests of the two passes that rewrite bytes in place, at every launch shape they choose, against plain references:
LZ00's keystream (keystream.cu: decode lifts it off the body, encode lays it over the body the LZSS encoder wrote) and BLZ's
byte reversal (decode_blz.cu: the encoder's source and its output).  Both launchers take gridDim.y = 32 below 148 streams,
8 below 1184 and 1 from there on, and stop gridDim.x at 4736 streams (blocks then stride over the streams), so the batch
sizes straddle every switch and the body lengths straddle the 256 x gridDim.y byte segments a block's threads cover.

References: the keystream restated in Python from the reference's ladder (tests/util.py), so a GPU-encoded LZ00 body XORed
with it must be the oracle's Lzss0 LZSS body of the same input; literal-only LZ00 files, whose every body byte reaches the
output; and for BLZ the oracle's bytes, which must decode back to the input."""
import numpy as np
import pytest

from auroralib.compression_b200 import layout, pack
from auroralib.compression_b200 import _abi as A
from tests.test_wrapped_encode_device_gpu import device_encode
from tests.util import literal_lzss0_body, lz00_file, lz00_stream_fast, xor_bytes

pytestmark = pytest.mark.gpu

BATCH_SIZES = [1, 147, 148, 1183, 1184, 4736, 4737, 6000]
LZSS0 = A.lz_props_window(0x1000, 0xF + 3, 3, 0xFEE)


def grid_y(n):
    return 1 if n >= 1184 else 8 if n >= 148 else 32


def lengths(n):
    """body lengths 0, 1, 255, 256, 257 and 256 x gridDim.y x k +- 1 for the shape n streams get; one batch of one stream
    per length at n = 1, plus a body above 1 MiB"""
    seg = 256 * grid_y(n)
    base = [0, 1, 255, 256, 257, seg - 1, seg + 1, 2 * seg - 1, 2 * seg + 1, 3 * seg]
    if n == 1:
        return [[v] for v in base + [(1 << 20) + 4099]]
    return [[base[i % len(base)] for i in range(n)]]


def literal_file(rng, body_len, key):
    """an LZ00 file whose body is body_len bytes of literals (a length of 1 mod 9 ends with an unread flag byte) -> (file, raw)"""
    k, r = divmod(body_len, 9)
    raw = rng.integers(0, 256, size=8 * k + max(r - 1, 0), dtype=np.uint8).tobytes()
    body = literal_lzss0_body(raw) + (b"\xff" if r == 1 else b"")
    assert len(body) == body_len
    return lz00_file(body, len(raw), key), raw


def device_decode(codec, fmt, comps, caps):
    import torch
    dev = torch.device("cuda", 0)
    base, off, ln = pack(comps)
    caps, doff, total = layout(caps)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a).astype(np.int64)).to(dev)
    d_src = torch.from_numpy(base).to(dev)
    before = d_src.clone()
    n = len(comps)
    d_dst = torch.full((total + 64,), 0xA5, dtype=torch.uint8, device=dev)
    d_olen, d_cons = torch.full((n,), -1, dtype=torch.int64, device=dev), torch.full((n,), -1, dtype=torch.int64, device=dev)
    d_st = torch.full((n,), -9, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    codec.decode_device(fmt, d_src, t(off), t(ln), d_dst, t(doff), t(caps), d_olen, d_cons, d_st)
    torch.cuda.synchronize(dev)
    assert torch.equal(d_src, before), "the device source changed"
    dst, olen = d_dst.cpu().numpy(), d_olen.cpu().numpy()
    outs = [dst[int(doff[i]):int(doff[i]) + min(int(olen[i]), int(caps[i]))].tobytes() for i in range(n)]
    return outs, olen.astype(np.uint64), d_cons.cpu().numpy().astype(np.uint64), d_st.cpu().numpy()


@pytest.mark.parametrize("n", BATCH_SIZES)
def test_lz00_decode_launch_shapes(codec, oracle, n):
    rng = np.random.default_rng(5000 + n)
    for lens in lengths(n):
        keys = [int(k) for k in rng.integers(0, 1 << 32, size=len(lens))]
        files, raws = zip(*[literal_file(rng, L, k) for L, k in zip(lens, keys)])
        caps = [len(r) for r in raws]
        ref, rlen, rcons, rst = oracle.decode_batch(A.FMT_LZ00, list(files), caps)
        assert (rst == A.OK).all() and list(ref) == list(raws)
        for where, (outs, olen, cons, st) in (("host", codec.decode_batch(A.FMT_LZ00, list(files), caps)),
                                              ("device", device_decode(codec, A.FMT_LZ00, list(files), caps))):
            bad = [i for i in range(len(files)) if st[i] != rst[i] or olen[i] != rlen[i] or cons[i] != rcons[i] or outs[i] != raws[i]]
            assert not bad, f"n={n} {where}: {len(bad)} streams differ; first #{bad[0]}: body {lens[bad[0]]} bytes, status {st[bad[0]]}"


def encode_inputs(rng, n):
    """incompressible inputs whose Lzss0 bodies (a flag byte per 8 literals) come out near the lengths of lengths(n)"""
    return [[rng.integers(0, 256, size=L * 8 // 9, dtype=np.uint8).tobytes() for L in lens] for lens in lengths(n)]


@pytest.mark.parametrize("n", BATCH_SIZES)
def test_lz00_encode_launch_shapes(codec, oracle, n):
    rng = np.random.default_rng(5100 + n)
    for raws in encode_inputs(rng, n):
        key = int(rng.integers(0, 1 << 32))
        opts = A.make_opts(quality=8, lz00_key=key)
        ref, rst = oracle.encode_batch(A.FMT_LZ00, raws, opts)
        lzss, _ = oracle.encode_batch(A.FMT_LZSS, raws, A.make_opts(quality=8, lzss=LZSS0))
        got, st = codec.encode_batch(A.FMT_LZ00, raws, opts)
        bad = np.nonzero((st != rst) | (st != A.OK))[0]
        assert not len(bad), f"n={n}: {len(bad)} statuses differ; first #{bad[0]}: {st[bad[0]]} / oracle {rst[bad[0]]}"
        for i, z in enumerate(got):
            assert z == ref[i], f"n={n}: stream #{i} ({len(raws[i])} bytes) differs from the oracle encoder"
            assert xor_bytes(z[64:], lz00_stream_fast(key, len(z) - 64)) == lzss[i][16:], f"n={n}: stream #{i}: keystream"
        caps = [codec.encode_bound(A.FMT_LZ00, len(r)) for r in raws]
        outs, dst, olen = device_encode(codec, A.FMT_LZ00, raws, caps, opts)
        bad = [i for i in range(len(raws)) if dst[i] != st[i] or outs[i] != got[i]]
        assert not bad, f"n={n}: device encode differs from the host in {len(bad)} streams; first #{bad[0]}: status {dst[bad[0]]}"


def test_lz00_encode_short_capacities(codec, oracle):
    """destinations shorter than the output: the keystream pass stops at the capacity (and starts 16 bytes into the core's
    output, under the header the wrapper writes)"""
    rng = np.random.default_rng(5200)
    raws = [rng.integers(0, 256, size=int(m), dtype=np.uint8).tobytes() for m in (0, 5, 300, 3000) for _ in range(8)]
    full, _ = oracle.encode_batch(A.FMT_LZ00, raws, A.make_opts(quality=8))
    caps = [max(0, len(z) + d) for z, d in zip(full, [-1, -17, -len(full[0]), 0, 16 - 64, 17 - 64, 63 - 64, 65 - 64] * 4)]
    base, off, ln = pack(raws)
    caps_a, doff, total = layout(caps)
    r_dst = np.zeros(total + 64, dtype=np.uint8)
    r_olen, r_st = oracle.encode_packed(A.FMT_LZ00, base, off, ln, r_dst, doff, caps_a, A.make_opts(quality=8))
    h_dst = np.zeros(total + 64, dtype=np.uint8)
    h_olen, h_st = codec.encode_packed(A.FMT_LZ00, base, off, ln, h_dst, doff, caps_a, A.make_opts(quality=8))
    # (the statuses are the oracle's; a core piece without room reports out_len 0 rather than the oracle's whole size)
    assert (h_st == r_st).all() and ((h_olen == r_olen) | (h_st == A.DST_TOO_SMALL)).all()
    assert (h_st == A.DST_TOO_SMALL).sum() >= 16
    outs, st, olen = device_encode(codec, A.FMT_LZ00, raws, caps, A.make_opts(quality=8))   # (bytes outside the windows: unchanged)
    assert (st == h_st).all() and (olen.astype(np.uint64) == h_olen).all()
    for i in range(len(raws)):
        if h_st[i] == A.OK:
            assert outs[i] == full[i]


@pytest.mark.parametrize("n", BATCH_SIZES)
def test_blz_encode_launch_shapes(codec, oracle, n):
    rng = np.random.default_rng(5300 + n)
    for lens in lengths(n):
        raws = [rng.integers(0, 256, size=L, dtype=np.uint8).tobytes() if i % 2 else bytes(rng.integers(0, 4, size=L, dtype=np.uint8))
                for i, L in enumerate(lens)]
        opts = A.make_opts(quality=8)
        got, st = codec.encode_batch(A.FMT_BLZ, raws, opts)
        ref, rst = oracle.encode_batch(A.FMT_BLZ, raws, opts)
        assert (st == rst).all()
        bad = [i for i in range(len(raws)) if got[i] != ref[i]]
        assert not bad, f"n={n}: {len(bad)} BLZ streams differ from the oracle; first #{bad[0]} ({len(raws[bad[0]])} bytes)"
        ok = [i for i in range(len(raws)) if st[i] == A.OK]
        outs, _, _, dst = oracle.decode_batch(A.FMT_BLZ, [got[i] for i in ok], [len(raws[i]) for i in ok])
        assert all(dst[j] == A.OK and outs[j] == raws[i] for j, i in enumerate(ok)), f"n={n}: a BLZ stream does not decode back"
