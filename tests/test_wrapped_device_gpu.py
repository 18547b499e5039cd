"""GPU tests of aurora_decode_batch_device for the wrapper formats (GCLZ, CXLZ, COMP, 3DS-LZ, LZ77, Level5, LZOn, Level5LZSS,
the LZSS-property family, SDPC, ECD, LZ00): on streams already in device memory, the same out_len / consumed / status and the
same destination bytes as the host entry point aurora_decode_batch on the same inputs, no host synchronisation (LZ77: one
read of its chunk count), and the launch counts the header promises."""
import numpy as np
import pytest

from auroralib.compression_b200 import AuroraError, layout, pack
from auroralib.compression_b200 import _abi as A
from tests.test_wrappers import _opt_sets
from tests.util import corrupt, fmt_id, synth

pytestmark = pytest.mark.gpu

WRAPPERS = A.WRAPPER_FORMATS
SENTINEL = 0xA5
# kernels per call (include/aurora_cuda.h): resolve + core + merge; + the store pass for the formats with stored bytes;
# LZ00: resolve, slot sizes, scan (2), keystream, core, merge; LZ77: resolve, scan (2), chunk fill, LZ10, LZ11, redo
# selection, redo LZ10, merge
LAUNCHES = {f: 3 for f in WRAPPERS} | {A.FMT_LEVEL5: 4, A.FMT_ECD: 4, A.FMT_LZ00: 7, A.FMT_LZ77: 9}
READS_BACK = (A.FMT_LZ77, A.FMT_LZ00)   # the calls that read one value back (LZ77: its chunk count; LZ00: its slot total)


def _device_inputs(comps, caps, dev, fill=SENTINEL):
    import torch
    base, off, ln = pack(comps)
    caps, doff, total = layout(caps)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a).astype(np.int64)).to(dev)
    d_src = torch.from_numpy(np.concatenate([base, np.zeros(16, np.uint8)])).to(dev)[:len(base)]
    n = len(comps)
    return dict(base=base, off=off, ln=ln, caps=caps, doff=doff, total=max(total, 16) + 64,
                d_src=d_src, d_off=t(off), d_len=t(ln), d_doff=t(doff), d_cap=t(caps),
                d_dst=torch.full((max(total, 16) + 64,), fill, dtype=torch.uint8, device=dev),
                d_olen=torch.full((n,), -1, dtype=torch.int64, device=dev),
                d_cons=torch.full((n,), -1, dtype=torch.int64, device=dev),
                d_st=torch.full((n,), -9, dtype=torch.int32, device=dev))


def _device_call(codec, fmt, X, opts=None, device=0, stream=None):
    codec.decode_device(fmt, X["d_src"], X["d_off"], X["d_len"], X["d_dst"], X["d_doff"], X["d_cap"], X["d_olen"], X["d_cons"],
                        X["d_st"], opts, device=device, stream=stream)


def _host(codec, fmt, X, opts=None):
    h_dst = np.full(X["total"], SENTINEL, dtype=np.uint8)
    olen, cons, st = codec.decode_packed(fmt, X["base"], X["off"], X["ln"], h_dst, X["doff"], X["caps"], opts)
    return h_dst, olen, cons, st


def _check_against_host(codec, fmt, X, opts, what):
    """the device results of X (already decoded) against the host entry point on the same inputs; whole buffers compared"""
    h_dst, olen, cons, st = _host(codec, fmt, X, opts)
    d_olen, d_cons, d_st = (X[k].cpu().numpy() for k in ("d_olen", "d_cons", "d_st"))
    bad = np.nonzero((d_st != st) | (d_olen.astype(np.uint64) != olen) | (d_cons.astype(np.uint64) != cons))[0]
    if len(bad):
        i = int(bad[0])
        pytest.fail(f"{fmt_id(fmt)} {what}: {len(bad)}/{len(st)} streams differ; first #{i}: status dev={d_st[i]} host={st[i]}, "
                    f"out_len {d_olen[i]}/{olen[i]}, consumed {d_cons[i]}/{cons[i]}, cap {X['caps'][i]}")
    d_dst = X["d_dst"].cpu().numpy()
    diff = np.nonzero(d_dst != h_dst)[0]
    if len(diff):
        j = int(diff[0])
        k = int(np.searchsorted(X["doff"].astype(np.int64), j, side="right")) - 1
        pytest.fail(f"{fmt_id(fmt)} {what}: {len(diff)} destination bytes differ; first at {j}, stream {k} "
                    f"(window at {X['doff'][k]}, out_len {olen[k]}, cap {X['caps'][k]}, status {st[k]})")
    return h_dst, olen, cons, st


def _run(codec, fmt, comps, caps, opts=None, what="", device=0):
    import torch
    dev = torch.device("cuda", device)
    X = _device_inputs(comps, caps, dev)
    torch.cuda.synchronize(dev)
    _device_call(codec, fmt, X, opts, device=device)
    torch.cuda.synchronize(dev)
    return _check_against_host(codec, fmt, X, opts, what)


def _parity(codec, oracle, fmt, seed, device=0):
    rng = np.random.default_rng(seed)
    for kw in _opt_sets(fmt):
        opts = A.make_opts(**({"quality": 8} | kw))
        raws = [synth(rng, int(rng.choice([1, 2, 7, 100, 1000, 4095, 4096, 4097, 9000, 40000, 70000])), i % 5) for i in range(48)]
        comps, st = oracle.encode_batch(fmt, raws, opts)
        keep = [i for i in range(len(raws)) if st[i] == 0]   # (ChunkLZ10 refuses chunks that end past 0xFFFF)
        raws, comps = [raws[i] for i in keep], [comps[i] for i in keep]
        _, olen, _, status = _run(codec, fmt, comps, [len(r) for r in raws], opts, f"valid {kw}", device)
        assert (status == A.OK).sum() >= len(raws) - (6 if fmt in (A.FMT_LZON, A.FMT_SDPC) else 0)
        bad = [corrupt(rng, c, i % 5) for i, c in enumerate(comps)]   # truncated / flipped / padded / empty / header-cut
        _run(codec, fmt, bad, [len(r) + int(rng.choice([0, 0, 64])) for r in raws], opts, f"fuzz {kw}", device)
        caps = [max(0, len(r) + int(rng.choice([-len(r), -17, -1, 0, 1, 100]))) for r in raws]   # 0, short, exact, larger
        _run(codec, fmt, comps, caps, opts, f"capacity {kw}", device)


@pytest.mark.parametrize("fmt", WRAPPERS, ids=fmt_id)
def test_matches_the_host(codec, oracle, fmt):
    _parity(codec, oracle, fmt, 8800 + fmt)


def test_lz77_mixed_sub_types_and_redo(codec, oracle, bmp):
    """LZ10, LZ11 and ChunkLZ10 streams in one batch (three core launches), with two chunked files cut inside their last chunk
    and chunked files whose chunk bodies are bit-flipped (the failing chunks the redo launch decodes once more)."""
    rng = np.random.default_rng(77)
    raws = [bmp[int(o):int(o) + int(n)] for o, n in zip(rng.integers(0, 900000, size=90), rng.integers(200, 30000, size=90))]
    types = [(0x10, 0), (0x11, 0), (0xF7, 0), (0xF7, 0x400)]
    comps = []
    for i, r in enumerate(raws):
        t, cs = types[i % 4]
        c, st = oracle.encode(A.FMT_LZ77, r, A.make_opts(quality=8, lz77_type=t, lz77_chunk_size=cs))
        assert st == 0
        comps.append(c)
    for k in (2, 6):
        comps[k] = comps[k][:len(comps[k]) - 40]
    for k in range(3, 90, 4):   # flip bytes inside the chunk bodies of the 1 KiB-chunk files
        b = bytearray(comps[k])
        for _ in range(3):
            b[int(rng.integers(len(b) // 2, len(b)))] ^= int(rng.integers(1, 256))
        comps[k] = bytes(b)
    caps = [len(r) for r in raws]
    _, _, _, st = _run(codec, A.FMT_LZ77, comps, caps, what="mixed")
    ref, rlen, rcons, rst = oracle.decode_batch(A.FMT_LZ77, comps, caps)
    assert (st == rst).all()
    assert sum(1 for i in range(90) if i % 4 != 3 and st[i] == A.OK) == 90 - 22 - 2


@pytest.mark.parametrize("fmt", [A.FMT_LEVEL5, A.FMT_ECD], ids=fmt_id)
def test_stored_and_compressed_alternate(codec, oracle, fmt):
    rng = np.random.default_rng(8500 + fmt)
    raws = [synth(rng, int(rng.choice([17, 100, 3000, 20000])), i % 5) for i in range(40)]
    comps = [oracle.encode(fmt, r, A.make_opts(quality=0 if i % 2 else 8))[0] for i, r in enumerate(raws)]
    h_dst, _, _, st = _run(codec, fmt, comps, [len(r) for r in raws], what="mixed")
    assert (st == A.OK).all()
    _, doff, _ = layout([len(r) for r in raws])
    assert all(h_dst[int(doff[i]):int(doff[i]) + len(r)].tobytes() == r for i, r in enumerate(raws))


def test_unsupported_sub_types(codec):
    blobs = [b"LZ77" + bytes([0x28, 4, 0, 0]) + bytes(16), b"LZ77" + bytes([0x30, 4, 0, 0]) + bytes(16), b"LZ77" + bytes([0x42, 4, 0, 0]) + bytes(16)]
    _, _, _, st = _run(codec, A.FMT_LZ77, blobs, [64] * 3, what="lz77 sub-types")
    assert (st == A.NOT_SUPPORTED).all()
    blobs = [(2 | (16 << 3)).to_bytes(4, "little") + bytes(16), (64).to_bytes(4, "little") + b"\x78\x9c" + bytes(16), bytes(4), bytes(5)]
    _, _, _, st = _run(codec, A.FMT_LEVEL5, blobs, [64] * 4, what="level5 sub-types")
    assert list(st[:2]) == [A.NOT_SUPPORTED] * 2


def test_lz00_keys_leave_the_source_unchanged(codec, oracle):
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(4000)
    raws = [synth(rng, int(rng.integers(1, 30000)), i % 5) for i in range(32)]
    for key in (0, 0xDEADBEEF):
        comps, st = oracle.encode_batch(A.FMT_LZ00, raws, A.make_opts(quality=8, lz00_key=key))
        assert (st == 0).all()
        X = _device_inputs(comps, [len(r) for r in raws], dev)
        before = X["d_src"].clone()
        torch.cuda.synchronize(dev)
        _device_call(codec, A.FMT_LZ00, X)
        torch.cuda.synchronize(dev)
        assert torch.equal(X["d_src"], before)
        h_dst, _, _, st = _check_against_host(codec, A.FMT_LZ00, X, None, f"key {key:#x}")
        assert (st == A.OK).all()
        assert all(h_dst[int(X["doff"][i]):int(X["doff"][i]) + len(r)].tobytes() == r for i, r in enumerate(raws))


def test_calls_are_stream_ordered_and_wait_only_to_read_back(codec, oracle):
    """every wrapper call launches what the header promises on the caller's stream; only LZ77 and LZ00, which read one
    value back, wait for that stream"""
    import torch
    dev = torch.device("cuda", 0)
    s = torch.cuda.Stream(device=dev)
    rng = np.random.default_rng(31)
    for fmt in WRAPPERS:
        kw = _opt_sets(fmt)[-1]
        opts = A.make_opts(**({"quality": 8} | kw))
        raws = [synth(rng, int(n), i % 5) for i, n in enumerate([100, 5000, 20000, 3000] * 4)]
        comps, st = oracle.encode_batch(fmt, raws, opts)
        caps = [len(r) for r in raws]
        X = _device_inputs(comps, caps, dev)
        h_src = X["d_src"].cpu().pin_memory()
        _device_call(codec, fmt, X, opts)   # the first call sizes the per-device scratch (a larger one is allocated once)
        torch.cuda.synchronize(dev)
        X["d_src"].zero_()
        X["d_dst"].fill_(SENTINEL)
        torch.cuda.synchronize(dev)
        with torch.cuda.stream(s):
            torch.cuda._sleep(1 << 29)   # ~0.3 s of GPU time: the stream is busy while the call below returns
            X["d_src"].copy_(h_src, non_blocking=True)
            before = codec.kernel_launches
            _device_call(codec, fmt, X, opts, stream=s.cuda_stream)
            assert codec.kernel_launches - before == LAUNCHES[fmt], fmt_id(fmt)
            if fmt not in READS_BACK:   # (they wait for the stream)
                assert not s.query(), f"{fmt_id(fmt)}: decode_device waited for the stream"
        s.synchronize()
        _check_against_host(codec, fmt, X, opts, "async")


def test_rejections(codec):
    import torch
    dev = torch.device("cuda", 0)
    comps = [b"GCLZ" + bytes(40)] * 4
    X = _device_inputs(comps, [64] * 4, dev)
    torch.cuda.synchronize(dev)
    before = codec.kernel_launches
    buf = torch.zeros(X["d_src"].numel() + 32, dtype=torch.uint8, device=dev)
    with pytest.raises(AuroraError):
        codec.decode_device(A.FMT_GCLZ, buf[1:1 + X["d_src"].numel()], X["d_off"], X["d_len"], X["d_dst"], X["d_doff"], X["d_cap"],
                            X["d_olen"], X["d_cons"], X["d_st"])
    with pytest.raises(AuroraError):
        _device_call(codec, A.FMT_LZ77, X, device=codec.device_count + 3)
    e = torch.empty(0, dtype=torch.int64, device=dev)
    codec.decode_device(A.FMT_LZ00, X["d_src"], e, e, X["d_dst"], e, e, e, e, torch.empty(0, dtype=torch.int32, device=dev))
    torch.cuda.synchronize(dev)
    assert codec.kernel_launches == before


def test_c2_shaped_gclz_and_chunklz10(codec):
    """4 096 files of 64 KiB from the C2 mix as GCLZ and as ChunkLZ10 with 4 KiB chunks, encoded by the engine: the device
    decode gives back the raw bytes."""
    import torch
    from auroralib.compression_b200 import corpus
    dev = torch.device("cuda", 0)
    n, size = 4096, 65536
    raw, _ = corpus.generate_mix(n, size, device=dev)
    raw_h = raw.reshape(n, size).cpu().numpy()
    raws = [raw_h[i].tobytes() for i in range(n)]
    for fmt, opts in ((A.FMT_GCLZ, A.make_opts(quality=8)), (A.FMT_LZ77, A.make_opts(quality=8, lz77_type=0xF7, lz77_chunk_size=0x1000))):
        comps, st = codec.encode_batch(fmt, raws, opts)
        keep = [i for i in range(n) if st[i] == 0]
        assert len(keep) >= n // 2, (fmt_id(fmt), len(keep))
        X = _device_inputs([comps[i] for i in keep], [size] * len(keep), dev)
        torch.cuda.synchronize(dev)
        _device_call(codec, fmt, X)
        torch.cuda.synchronize(dev)
        assert (X["d_st"] == 0).all() and (X["d_olen"] == size).all() and torch.equal(X["d_cons"], X["d_len"])
        want = raw.reshape(n, size)[torch.tensor(keep, device=dev)]
        got = X["d_dst"][:len(keep) * size].reshape(len(keep), size)
        assert torch.equal(got, want), fmt_id(fmt)


def test_second_device(codec, oracle):
    if codec.device_count < 2:
        pytest.skip("one device in the context")
    for fmt in (A.FMT_GCLZ, A.FMT_LZ77, A.FMT_ECD, A.FMT_LZ00):
        _parity(codec, oracle, fmt, 9900 + fmt, device=1)
