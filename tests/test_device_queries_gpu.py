"""GPU tests of the device-resident GetDecompressedSize, IsMatch and offset-scan entry points and of
BatchCodec.decode_device_sized: the same answers as the host entry points on streams already in device memory, no host
synchronisation inside the calls, and the launch counts the header promises."""
import re

import numpy as np
import pytest

from auroralib.compression_b200 import AuroraError, pack
from auroralib.compression_b200 import _abi as A
from tests.util import ALL_FORMATS, MATCHABLE, SIZED_FORMATS, corrupt, decoded_size_blobs, fmt_id, is_match_blobs, rom_like_image, synth

pytestmark = pytest.mark.gpu

BYTE_LZ = [f for f in ALL_FORMATS if f not in SIZED_FORMATS]
SCAN_FORMATS = [f for f in ALL_FORMATS if f not in (A.FMT_LZ4_BLOCK, A.FMT_SNAPPY_BLOCK, A.FMT_BLZ)]
ORDERS = (A.ENDIAN_DEFAULT, A.ENDIAN_LITTLE, A.ENDIAN_BIG)


def _to_device(blobs, align, dev, shift=0):
    """Pack blobs at `align`-byte offsets into one CUDA tensor that starts `shift` bytes into its allocation."""
    import torch
    base, off, ln = pack(blobs, align)
    buf = torch.zeros(len(base) + shift + 16, dtype=torch.uint8, device=dev)
    buf[shift:shift + len(base)] = torch.from_numpy(base).to(dev)
    d_src = buf[shift:shift + len(base)]
    return d_src, torch.from_numpy(off.astype(np.int64)).to(dev), torch.from_numpy(ln.astype(np.int64)).to(dev)


def _sizes_on_device(codec, fmt, blobs, opts, size_scan, device, dev):
    import torch
    d_src, d_off, d_len = _to_device(blobs, 16, dev)
    n = len(blobs)
    d_size = torch.full((n,), 12345, dtype=torch.int64, device=dev)
    d_st = torch.full((n,), -1, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    codec.decoded_size_device(fmt, d_src, d_off, d_len, d_size, d_st, opts, size_scan=size_scan, device=device)
    torch.cuda.synchronize(dev)
    return d_size.cpu().numpy().astype(np.uint64), d_st.cpu().numpy()


def _check_sizes(codec, oracle, fmt, device=0):
    import torch
    dev = torch.device("cuda", device)
    blobs = decoded_size_blobs(oracle, fmt)
    for order in ORDERS:
        opts = A.make_opts(byte_order=order)
        for scan in (False, True):
            size, st = _sizes_on_device(codec, fmt, blobs, opts, scan, device, dev)
            h_size, h_st = codec.decoded_size_batch(fmt, blobs, opts, size_scan=scan)
            bad = np.nonzero((size != h_size) | (st != h_st))[0]
            assert not len(bad), (fmt_id(fmt), order, scan, int(bad[0]), int(size[bad[0]]), int(st[bad[0]]), int(h_size[bad[0]]), int(h_st[bad[0]]))
            valid = 0
            for i, b in enumerate(blobs):
                rs, rst = oracle.decoded_size(fmt, b, opts, 1 if scan else 0)
                if rst == A.OK:
                    valid += 1
                    assert (int(size[i]), int(st[i])) == (rs, rst), (fmt_id(fmt), order, scan, i)
            if fmt in BYTE_LZ and not scan:
                assert (st == A.NOT_SUPPORTED).all() and (size == 0).all()
            else:
                assert valid > 0


def _check_is_match(codec, oracle, bmp, fmt, device=0):
    import torch
    dev = torch.device("cuda", device)
    blobs = is_match_blobs(oracle, bmp, fmt)
    host = codec.is_match_batch(fmt, blobs)
    ref = np.array([oracle.is_match(fmt, b) for b in blobs])
    assert (host == ref).all()
    for align, shift in ((16, 0), (1, 3)):
        d_src, d_off, d_len = _to_device(blobs, align, dev, shift)
        d_m = torch.full((len(blobs),), 7, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        codec.is_match_device(fmt, d_src, d_off, d_len, d_m, device=device)
        torch.cuda.synchronize(dev)
        got = d_m.cpu().numpy()
        assert set(np.unique(got).tolist()) <= {0, 1}
        bad = np.nonzero(got.astype(bool) != host)[0]
        assert not len(bad), (fmt_id(fmt), align, int(bad[0]), blobs[int(bad[0])][:24].hex())


def _check_scan(codec, oracle, bmp, fmt, device=0):
    import torch
    dev = torch.device("cuda", device)
    rng = np.random.default_rng(91 + fmt)
    image, _ = rom_like_image(oracle, rng, fmt, [bmp[2000:12000], bytes(2000), synth(rng, 4000, 0), synth(rng, 3000, 2)])
    host = codec.scan_offsets(fmt, image)
    for shift in (0, 5):
        buf = torch.zeros(len(image) + shift, dtype=torch.uint8, device=dev)
        buf[shift:] = torch.frombuffer(bytearray(image), dtype=torch.uint8).to(dev)
        d_m = torch.full((len(image),), 7, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        codec.scan_offsets_device(fmt, buf[shift:], d_m, device=device)
        torch.cuda.synchronize(dev)
        got = d_m.cpu().numpy()
        bad = np.nonzero(got.astype(bool) != host)[0]
        assert not len(bad) and set(np.unique(got).tolist()) <= {0, 1}, (fmt_id(fmt), shift, bad[:4])


# ---- 1-3: the same answers as the host entry points
@pytest.mark.parametrize("fmt", ALL_FORMATS, ids=fmt_id)
def test_sizes_match_the_host(codec, oracle, fmt):
    _check_sizes(codec, oracle, fmt)


@pytest.mark.parametrize("fmt", MATCHABLE, ids=fmt_id)
def test_is_match_matches_the_host(codec, oracle, bmp, fmt):
    _check_is_match(codec, oracle, bmp, fmt)


@pytest.mark.parametrize("fmt", SCAN_FORMATS, ids=fmt_id)
def test_scan_matches_the_host(codec, oracle, bmp, fmt):
    _check_scan(codec, oracle, bmp, fmt)


# ---- 4: rejections launch nothing
def _rejected(codec, call, host_name=None):
    before = codec.kernel_launches
    with pytest.raises(AuroraError, match="INVALID_ARGUMENT") as e:
        call()
    assert codec.kernel_launches == before
    if host_name:   # the last error names the host entry point that takes the format
        assert re.search(host_name + r"\b(?!_device)", str(e.value)), str(e.value)


def test_rejections(codec, oracle):
    import torch
    dev = torch.device("cuda", 0)
    blobs = [oracle.encode(A.FMT_LZ10, bytes(range(200)) * 4)[0]] * 3
    d_src, d_off, d_len = _to_device(blobs, 16, dev)
    d_size = torch.zeros(3, dtype=torch.int64, device=dev)
    d_st = torch.zeros(3, dtype=torch.int32, device=dev)
    d_m = torch.zeros(64, dtype=torch.uint8, device=dev)
    for fmt in (A.FMT_GCLZ, A.FMT_LZ77, A.FMT_LZ00, 99):
        for scan in (False, True):
            _rejected(codec, lambda: codec.decoded_size_device(fmt, d_src, d_off, d_len, d_size, d_st, size_scan=scan),
                      "aurora_decoded_size_batch" if fmt != 99 else None)
    for fmt in (A.FMT_GCLZ, A.FMT_LEVEL5, A.FMT_LZ4_BLOCK, A.FMT_SNAPPY_BLOCK, 99):
        _rejected(codec, lambda: codec.is_match_device(fmt, d_src, d_off, d_len, d_m), "aurora_is_match_batch")
    for fmt in (A.FMT_BLZ, A.FMT_GCLZ, A.FMT_LZ4_BLOCK, A.FMT_SNAPPY_BLOCK, 99):
        _rejected(codec, lambda: codec.scan_offsets_device(fmt, d_m, d_m), "aurora_scan_offsets")
    for device in (-1, codec.device_count):
        _rejected(codec, lambda: codec.decoded_size_device(A.FMT_LZ10, d_src, d_off, d_len, d_size, d_st, device=device))
        _rejected(codec, lambda: codec.is_match_device(A.FMT_LZ10, d_src, d_off, d_len, d_m, device=device))
        _rejected(codec, lambda: codec.scan_offsets_device(A.FMT_LZ10, d_m, d_m, device=device))
    # the size entry point stages a size scan like decode: its source must start 16-byte aligned, with or without a scan
    big = torch.zeros(d_src.numel() + 32, dtype=torch.uint8, device=dev)
    for fmt, scan in ((A.FMT_LZ10, False), (A.FMT_LZ4, True)):
        _rejected(codec, lambda: codec.decoded_size_device(fmt, big[1:1 + d_src.numel()], d_off, d_len, d_size, d_st, size_scan=scan))
    with pytest.raises(AuroraError, match="16-byte aligned"):
        codec.decode_device_sized(A.FMT_LZ10, big[8:8 + d_src.numel()], d_off, d_len)
    # empty batches are accepted and launch nothing
    before = codec.kernel_launches
    e64 = torch.zeros(0, dtype=torch.int64, device=dev)
    codec.decoded_size_device(A.FMT_LZ4, d_src, e64, e64, e64, torch.zeros(0, dtype=torch.int32, device=dev), size_scan=True)
    codec.is_match_device(A.FMT_LZ10, d_src, e64, e64, d_m[:0])
    codec.scan_offsets_device(A.FMT_LZ10, d_m[:0], d_m)
    assert codec.kernel_launches == before


# ---- 5: asynchronous and ordered on the caller's stream
def test_calls_are_asynchronous_and_stream_ordered(codec, oracle, bmp):
    import torch
    dev = torch.device("cuda", 0)
    s = torch.cuda.Stream(device=dev)
    cases = [(A.FMT_LZ10, False, 1), (A.FMT_YAZ0, True, 1), (A.FMT_LZ4, False, 1), (A.FMT_LZ4, True, 2), (A.FMT_PRS, True, 2)]
    for fmt, scan, launches in cases:
        blobs = decoded_size_blobs(oracle, fmt)
        base, off, ln = pack(blobs)
        h_src = torch.from_numpy(base).pin_memory()
        d_src = torch.zeros(len(base), dtype=torch.uint8, device=dev)
        d_off = torch.from_numpy(off.astype(np.int64)).to(dev)
        d_len = torch.from_numpy(ln.astype(np.int64)).to(dev)
        d_size = torch.full((len(blobs),), 3, dtype=torch.int64, device=dev)
        d_st = torch.full((len(blobs),), -1, dtype=torch.int32, device=dev)
        torch.cuda.synchronize(dev)
        with torch.cuda.stream(s):
            torch.cuda._sleep(1 << 29)   # ~0.3 s of GPU time: the stream is busy while the calls below return
            d_src.copy_(h_src, non_blocking=True)
            before = codec.kernel_launches
            codec.decoded_size_device(fmt, d_src, d_off, d_len, d_size, d_st, size_scan=scan, stream=s.cuda_stream)
            assert codec.kernel_launches - before == launches
            assert not s.query(), "decoded_size_device waited for the stream"
        s.synchronize()
        h_size, h_st = codec.decoded_size_batch(fmt, blobs, size_scan=scan)
        assert (d_size.cpu().numpy().astype(np.uint64) == h_size).all() and (d_st.cpu().numpy() == h_st).all(), (fmt_id(fmt), scan)

    blobs = is_match_blobs(oracle, bmp, A.FMT_LZ10)
    base, off, ln = pack(blobs, 1)
    h_src = torch.from_numpy(base).pin_memory()
    d_src = torch.zeros(len(base), dtype=torch.uint8, device=dev)
    d_off = torch.from_numpy(off.astype(np.int64)).to(dev)
    d_len = torch.from_numpy(ln.astype(np.int64)).to(dev)
    d_m = torch.full((len(blobs),), 7, dtype=torch.uint8, device=dev)
    rng = np.random.default_rng(5)
    image, _ = rom_like_image(oracle, rng, A.FMT_LZ10, [bmp[:6000], synth(rng, 3000, 1)])
    h_img = torch.frombuffer(bytearray(image), dtype=torch.uint8).pin_memory()
    d_img = torch.zeros(len(image), dtype=torch.uint8, device=dev)
    d_scan = torch.full((len(image),), 7, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    with torch.cuda.stream(s):
        torch.cuda._sleep(1 << 29)
        d_src.copy_(h_src, non_blocking=True)
        d_img.copy_(h_img, non_blocking=True)
        before = codec.kernel_launches
        codec.is_match_device(A.FMT_LZ10, d_src, d_off, d_len, d_m, stream=s.cuda_stream)
        assert codec.kernel_launches - before == 1
        codec.scan_offsets_device(A.FMT_LZ10, d_img, d_scan, stream=s.cuda_stream)
        assert codec.kernel_launches - before == 2
        assert not s.query(), "the IsMatch / scan calls waited for the stream"
    s.synchronize()
    assert (d_m.cpu().numpy().astype(bool) == codec.is_match_batch(A.FMT_LZ10, blobs)).all()
    assert (d_scan.cpu().numpy().astype(bool) == codec.scan_offsets(A.FMT_LZ10, image)).all()


# ---- 6: decode_device_sized
def _forged(codec, fmt, comp, max_size):
    """The stream with 4 bytes of its header (or BLZ footer) overwritten so that its size peek claims more than max_size."""
    for p in list(range(0, min(16, len(comp) - 4))) + [len(comp) - 4]:
        b = bytearray(comp)
        b[p:p + 4] = b"\xff\xff\xff\x7f"
        size, st = codec.decoded_size_batch(fmt, [bytes(b)])
        if st[0] == A.OK and int(size[0]) > max_size:
            return bytes(b)
    raise AssertionError(f"{fmt_id(fmt)}: no forged header found")


@pytest.mark.parametrize("fmt", ALL_FORMATS, ids=fmt_id)
def test_decode_device_sized_matches_the_host(codec, oracle, fmt):
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(700 + fmt)
    max_size = 5000   # below the largest raw stream: a valid stream whose size is over the limit gets no capacity
    raws = [synth(rng, int(rng.integers(1, 7000)), i % 5) for i in range(40)] + [b"", bytes(1)]
    comps, st = oracle.encode_batch(fmt, raws, A.make_opts(quality=8))
    keep = [i for i in range(len(raws)) if st[i] == 0]
    raws, comps = [raws[i] for i in keep], [comps[i] for i in keep]
    # ground truth where the reference round-trips (not every format represents an empty input, and the reference's PRS
    # encoder writes a few random-data streams its decoder reads differently)
    ref, _, _, rst = oracle.decode_batch(fmt, comps, [len(r) for r in raws])
    blobs, truth = list(comps), [r if rst[i] == A.OK and ref[i] == r else None for i, r in enumerate(raws)]
    assert sum(t is not None for t in truth) >= len(raws) * 3 // 4
    for i, c in enumerate(comps[:24]):
        blobs.append(corrupt(rng, c, i % 5))
        truth.append(None)
    if fmt in SIZED_FORMATS:
        blobs += [_forged(codec, fmt, comps[i], max_size) for i in range(3)]
        truth += [None] * 3
    size_scan = True
    sizes, sst = codec.decoded_size_batch(fmt, blobs, size_scan=size_scan)
    caps = np.where((sst == A.OK) & (sizes <= max_size), sizes, 0).astype(np.uint64)
    h_outs, h_olen, h_cons, h_st = codec.decode_batch(fmt, blobs, caps)

    d_src, d_off, d_len = _to_device(blobs, 16, dev)
    s = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize(dev)
    d_dst, d_doff, d_cap, d_olen, d_cons, d_st = codec.decode_device_sized(fmt, d_src, d_off, d_len, size_scan=size_scan,
                                                                           max_size=max_size, stream=s.cuda_stream)
    s.synchronize()
    assert (d_cap.cpu().numpy().astype(np.uint64) == caps).all()
    doff = d_doff.cpu().numpy()
    assert (doff % 16 == 0).all() and (np.diff(doff) >= (caps[:-1].astype(np.int64) + 15) // 16 * 16).all()
    olen, cons, stt = d_olen.cpu().numpy().astype(np.uint64), d_cons.cpu().numpy().astype(np.uint64), d_st.cpu().numpy()
    assert (stt == h_st).all() and (olen == h_olen).all() and (cons == h_cons).all(), fmt_id(fmt)
    dst = d_dst.cpu().numpy()
    for i in range(len(blobs)):
        got = dst[int(doff[i]):int(doff[i]) + min(int(olen[i]), int(caps[i]))].tobytes()
        assert got == h_outs[i], (fmt_id(fmt), i)
        if truth[i] is not None and len(truth[i]) <= max_size:
            assert stt[i] == A.OK and got == truth[i], (fmt_id(fmt), i)
    assert any(t is not None and len(t) > max_size for t in truth)   # the over-limit case was exercised
    assert (stt[[i for i, t in enumerate(truth) if t is not None and len(t) > max_size]] != A.OK).all()


def test_decode_device_sized_c2_shape(codec):
    """4 096 LZ10 streams of 64 KiB from the C2 mix, encoded by the engine, decoded with sizes found on the device."""
    import torch
    import bench
    from auroralib.compression_b200 import corpus
    dev = torch.device("cuda", 0)
    n, size = 4096, 65536
    raw, _ = corpus.generate_mix(n, size, device=dev)
    raw = raw.reshape(-1)
    r_len = torch.full((n,), size, dtype=torch.int64, device=dev)
    r_off = torch.arange(n, dtype=torch.int64, device=dev) * size
    ts = torch.cuda.Stream(device=dev)
    packed, p_off, c_len, _, _ = bench.gpu_encode(codec, A.FMT_LZ10, raw, r_off, r_len, A.make_opts(quality=8), dev, ts)
    d_dst, d_doff, d_cap, d_olen, d_cons, d_st = codec.decode_device_sized(A.FMT_LZ10, packed, p_off, c_len, stream=ts.cuda_stream)
    ts.synchronize()
    assert (d_st == 0).all() and (d_olen == size).all() and (d_cap == size).all() and (d_cons == c_len).all()
    assert torch.equal(d_doff, r_off)
    assert torch.equal(d_dst[:n * size], raw)


# ---- 7: a second device
def test_second_device(codec, oracle, bmp):
    if codec.device_count < 2:
        pytest.skip("one device in the context")
    for fmt in (A.FMT_LZ10, A.FMT_YAZ0, A.FMT_BLZ, A.FMT_LZ4, A.FMT_PRS):
        _check_sizes(codec, oracle, fmt, device=1)
    for fmt in (A.FMT_LZ10, A.FMT_LZ11, A.FMT_PRS, A.FMT_YAZ0, A.FMT_BLZ):
        _check_is_match(codec, oracle, bmp, fmt, device=1)
    for fmt in (A.FMT_LZ10, A.FMT_PRS, A.FMT_LZ4):
        _check_scan(codec, oracle, bmp, fmt, device=1)
