"""GPU tests of aurora_encode_batch_device for the wrapper formats (GCLZ, CXLZ, COMP, 3DS-LZ, LZ77 with ChunkLZ10, Level5, LZOn,
Level5LZSS, the LZSS-property family, SDPC, ECD, LZ00): on sources already in device memory, the same out_len / status as the
host entry point aurora_encode_batch, the same bytes for OK streams (and the oracle's), nothing written outside the
destination windows, the caller's source untouched, no host synchronisation (ChunkLZ10: one read of its chunk count), and
the launch counts the header promises."""
import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests.test_encode_edges_gpu import host_encode
from tests.test_wrap_encode_rule_simt import LEVEL5_EMPTY, opt_sets
from tests.test_wrappers import _opt_sets
from tests.util import fmt_id, synth

pytestmark = pytest.mark.gpu

WRAPPERS = A.WRAPPER_FORMATS
SENTINEL = 0xEE
LENGTHS = [0, 1, 16, 17, 100, 4096, 4097, 20000, 70000]


def launches(fmt, kw):
    """kernels per call (include/aurora_cuda.h): plan + core + finish; + the keystream pass for LZ00; ChunkLZ10: plan, scan
    (2), chunk fill, core, finish"""
    if fmt == A.FMT_LZ77 and kw.get("lz77_type") == 0xF7:
        return 6
    return 4 if fmt == A.FMT_LZ00 else 3


def roomy(n):
    """a capacity every wrapper encode of n bytes fits, ChunkLZ10 chunk slots of any chunk size >= 0x400 included"""
    return 8 + 2 * (n + 2) + 3 * n + 70 * (n // 0x400 + 2) + 1024


def _device_inputs(raws, caps, dev):
    import torch
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
    t64 = lambda v: torch.tensor(v, dtype=torch.int64, device=dev)
    return dict(doff=doff, caps=list(caps), d_src=torch.from_numpy(src).to(dev), d_off=t64(soff), d_len=t64([len(r) for r in raws]),
                d_dst=torch.full((pos + 32,), SENTINEL, dtype=torch.uint8, device=dev), d_doff=t64(doff), d_cap=t64(list(caps)),
                d_olen=torch.full((len(raws),), -1, dtype=torch.int64, device=dev),
                d_st=torch.full((len(raws),), 77, dtype=torch.int32, device=dev))


def _call(codec, fmt, X, opts, device=0, stream=None):
    codec.encode_device(fmt, X["d_src"], X["d_off"], X["d_len"], X["d_dst"], X["d_doff"], X["d_cap"], X["d_olen"], X["d_st"], opts,
                        device=device, stream=stream)


def _results(fmt, X):
    """(window bytes [0, min(out_len, cap)), status, out_len); nothing outside the windows changed"""
    dst = X["d_dst"].cpu().numpy()
    out_len, status = X["d_olen"].cpu().numpy(), X["d_st"].cpu().numpy()
    inside = np.zeros(len(dst), dtype=bool)
    for o, c in zip(X["doff"], X["caps"]):
        inside[o:o + c] = True
    assert (dst[~inside] == SENTINEL).all(), f"{fmt_id(fmt)}: bytes outside the destination windows changed"
    return [dst[o:o + min(int(l), c)].tobytes() for o, c, l in zip(X["doff"], X["caps"], out_len)], status, out_len


def device_encode(codec, fmt, raws, caps, opts, device=0):
    import torch
    dev = torch.device("cuda", device)
    X = _device_inputs(raws, caps, dev)
    before = X["d_src"].clone()
    torch.cuda.synchronize(dev)
    _call(codec, fmt, X, opts, device=device)
    torch.cuda.synchronize(dev)
    assert torch.equal(X["d_src"], before), f"{fmt_id(fmt)}: the source changed"
    return _results(fmt, X)


def _oracle_ref(oracle, fmt, raw, kw, opts):
    if fmt == A.FMT_LEVEL5 and not raw and kw.get("quality", 8) != 0:
        return LEVEL5_EMPTY, A.OK   # (the oracle cannot encode an empty Level5 stream)
    return oracle.encode(fmt, raw, opts)


def _same_as_host(codec, fmt, raws, caps, opts, what, device=0):
    hgot, hst, hlen = host_encode(codec, fmt, raws, caps, opts)
    dgot, dst, dlen = device_encode(codec, fmt, raws, caps, opts, device)
    bad = [i for i in range(len(raws)) if hst[i] != dst[i] or int(hlen[i]) != int(dlen[i]) or (hst[i] == A.OK and hgot[i] != dgot[i])]
    if bad:
        i = bad[0]
        pytest.fail(f"{fmt_id(fmt)} {what}: {len(bad)}/{len(raws)} streams differ; first #{i} (len {len(raws[i])}, cap {caps[i]}): "
                    f"status dev={dst[i]} host={hst[i]}, out_len {dlen[i]}/{hlen[i]}, bytes equal {hgot[i] == dgot[i]}")
    return dgot, dst, dlen


def _raws(seed, lengths=LENGTHS):
    rng = np.random.default_rng(seed)
    out = []
    for i, n in enumerate(lengths):
        out.append(synth(rng, n, i % 4))
        if n >= 16:
            out.append(rng.integers(0, 256, size=n, dtype=np.uint8).tobytes())   # incompressible
    return out


@pytest.mark.parametrize("fmt", WRAPPERS, ids=fmt_id)
@pytest.mark.parametrize("quality", [0, 8])
def test_matches_the_host_and_the_oracle(codec, oracle, fmt, quality):
    raws = _raws(5100 + fmt)
    for kw in opt_sets(fmt):
        kw = kw | {"quality": quality} if "quality" not in kw else kw
        opts = A.make_opts(**kw)
        got, st, _ = _same_as_host(codec, fmt, raws, [roomy(len(r)) for r in raws], opts, f"q{quality} {kw}")
        if kw.get("lz77_type") == 0x28 or (kw.get("level5_type") == 2 and kw["quality"] != 0):
            assert (st == A.NOT_SUPPORTED).all()
            continue
        for i, r in enumerate(raws):
            ref, rst = _oracle_ref(oracle, fmt, r, kw, opts)
            if rst == A.OK and st[i] == A.OK:
                assert got[i] == ref, (fmt_id(fmt), kw, len(r))
            if fmt != A.FMT_LZ77:   # (ChunkLZ10 refuses chunks that end past 0xFFFF; the oracle too)
                assert st[i] == rst or (fmt == A.FMT_ECD and rst == A.INVALID_ARGUMENT), (fmt_id(fmt), kw, len(r), int(st[i]), rst)


@pytest.mark.parametrize("fmt", WRAPPERS, ids=fmt_id)
def test_capacity_sweep(codec, fmt):
    """the host's needed size, one below it, inside the header and 0: status and out_len as on the host"""
    raws = _raws(5300 + fmt, [17, 100, 4097, 20000])
    for kw in _opt_sets(fmt):
        opts = A.make_opts(**({"quality": 8} | kw))
        _, hst, hlen = host_encode(codec, fmt, raws, [roomy(len(r)) for r in raws], opts)
        assert (hst == A.OK).sum() >= len(raws) - 2
        rs, caps = [], []
        for r, s, need in zip(raws, hst, hlen):
            if s != A.OK:
                continue
            for c in (int(need), int(need) - 1, 7, 3, 0):
                rs.append(r)
                caps.append(max(c, 0))
        _same_as_host(codec, fmt, rs, caps, opts, f"capacities {kw}")


def test_chunklz10_compaction_and_table_limit(codec, oracle, bmp):
    """ChunkLZ10 with 0x400 and 0x1000 chunks on compressible data (every chunk lands on an earlier chunk's slot), files of one
    chunk, and incompressible files whose end offsets pass 0xFFFF"""
    rng = np.random.default_rng(91)
    comp = [bmp[int(o):int(o) + int(n)] for o, n in zip(rng.integers(0, 900000, size=40), rng.integers(3000, 30000, size=40))]
    one = [bmp[1000:1000 + n] for n in (1, 100, 0x3FF, 0x400)]
    noise = [rng.integers(0, 256, size=n, dtype=np.uint8).tobytes() for n in (0x10000, 70000, 100000)]
    for chunk in (0x400, 0x1000):
        kw = dict(quality=8, lz77_type=0xF7, lz77_chunk_size=chunk)
        opts = A.make_opts(**kw)
        raws = comp + one + noise
        got, st, _ = _same_as_host(codec, A.FMT_LZ77, raws, [roomy(len(r)) for r in raws], opts, f"chunk {chunk:#x}")
        for i, r in enumerate(raws):
            ref, rst = oracle.encode(A.FMT_LZ77, r, opts)
            assert st[i] == rst and (rst != A.OK or got[i] == ref), (chunk, len(r), int(st[i]), rst)
        assert (st[:len(comp) + len(one)] == A.OK).sum() >= len(comp) and (st[-2:] == A.INVALID_ARGUMENT).all()


@pytest.mark.parametrize("fmt", [A.FMT_LEVEL5, A.FMT_ECD], ids=fmt_id)
def test_stored_and_compressed_alternate(codec, oracle, fmt):
    """ECD streams of 16 bytes or less and ones whose body does not shrink are stored, the others compressed, in one batch;
    Level5 at quality 0 stores everything, at quality 8 nothing"""
    rng = np.random.default_rng(8600 + fmt)
    raws = []
    for i in range(60):
        n = int(rng.choice([5, 16, 17, 100, 3000, 20000]))
        raws.append(synth(rng, n, 0) if i % 2 else rng.integers(0, 256, size=n, dtype=np.uint8).tobytes())
    for q in (0, 8):
        opts = A.make_opts(quality=q)
        got, st, _ = _same_as_host(codec, fmt, raws, [roomy(len(r)) for r in raws], opts, f"q{q}")
        assert (st == A.OK).all()
        assert all(got[i] == oracle.encode(fmt, r, opts)[0] for i, r in enumerate(raws))
        if fmt == A.FMT_ECD and q == 8:
            flags = {g[3] for g in got}
            assert flags == {0, 1}


def test_level5_past_16_mib(codec):
    """Above 0xFFFFFF bytes LZ10 writes its 8-byte header: the body moves down by 4 (compared with the host entry point)"""
    rng = np.random.default_rng(5)
    raws = [synth(rng, (1 << 24) + 4096, 0), synth(rng, 5000, 1)]
    _, st, _ = _same_as_host(codec, A.FMT_LEVEL5, raws, [roomy(len(r)) for r in raws], A.make_opts(quality=2), "16 MiB")
    assert (st == A.OK).all()


@pytest.mark.parametrize("fmt", WRAPPERS, ids=fmt_id)
def test_round_trip(codec, fmt):
    import torch
    dev = torch.device("cuda", 0)
    raws = _raws(5500 + fmt, [1, 100, 4097, 20000, 70000])
    for kw in _opt_sets(fmt):
        opts = A.make_opts(**({"quality": 8} | kw))
        X = _device_inputs(raws, [roomy(len(r)) for r in raws], dev)
        _call(codec, fmt, X, opts)
        torch.cuda.synchronize(dev)
        ok = (X["d_st"] == A.OK).cpu().numpy()
        if fmt == A.FMT_LZ77 and kw.get("lz77_type") == 0xF7:
            assert ok.sum() >= len(raws) - 2
        else:
            assert ok.all(), (fmt_id(fmt), kw, X["d_st"].cpu().numpy())
        keep = np.nonzero(ok)[0]
        d_dst, d_doff, d_olen = X["d_dst"], X["d_doff"][keep], X["d_olen"][keep]
        caps = [len(raws[i]) for i in keep]
        doff, pos = [], 0
        for c in caps:
            doff.append(pos)
            pos += ((c + 15) & ~15) + 16
        out = torch.zeros(pos + 16, dtype=torch.uint8, device=dev)
        t64 = lambda v: torch.tensor(v, dtype=torch.int64, device=dev)
        k = len(keep)
        o_len, o_cons = torch.zeros(k, dtype=torch.int64, device=dev), torch.zeros(k, dtype=torch.int64, device=dev)
        o_st = torch.zeros(k, dtype=torch.int32, device=dev)
        codec.decode_device(fmt, d_dst, d_doff, d_olen, out, t64(doff), t64(caps), o_len, o_cons, o_st, opts)
        torch.cuda.synchronize(dev)
        assert (o_st == A.OK).all(), (fmt_id(fmt), kw)
        h = out.cpu().numpy()
        assert all(h[doff[j]:doff[j] + caps[j]].tobytes() == raws[i] for j, i in enumerate(keep)), (fmt_id(fmt), kw)


def test_calls_are_asynchronous_and_stream_ordered(codec):
    import torch
    dev = torch.device("cuda", 0)
    s = torch.cuda.Stream(device=dev)
    rng = np.random.default_rng(32)
    raws = [synth(rng, int(n), i % 5) for i, n in enumerate([100, 5000, 20000, 3000] * 4)]
    for fmt in WRAPPERS:
        kw = {"quality": 8} | _opt_sets(fmt)[-1]
        opts = A.make_opts(**kw)
        caps = [roomy(len(r)) for r in raws]
        X = _device_inputs(raws, caps, dev)
        h_src = X["d_src"].cpu().pin_memory()
        _call(codec, fmt, X, opts)   # the first call sizes the per-device scratch (a larger one is allocated once)
        torch.cuda.synchronize(dev)
        X["d_src"].zero_()
        X["d_dst"].fill_(SENTINEL)
        torch.cuda.synchronize(dev)
        with torch.cuda.stream(s):
            torch.cuda._sleep(1 << 29)   # ~0.3 s of GPU time: the stream is busy while the call below returns
            X["d_src"].copy_(h_src, non_blocking=True)
            before = codec.kernel_launches
            _call(codec, fmt, X, opts, stream=s.cuda_stream)
            assert codec.kernel_launches - before == launches(fmt, kw), fmt_id(fmt)
            if not (fmt == A.FMT_LZ77 and kw.get("lz77_type") == 0xF7):   # (ChunkLZ10 reads its chunk count back)
                assert not s.query(), f"{fmt_id(fmt)}: encode_device waited for the stream"
        s.synchronize()
        dgot, dst, dlen = _results(fmt, X)
        hgot, hst, hlen = host_encode(codec, fmt, raws, caps, opts)
        assert (hst == dst).all() and (hlen == dlen.astype(np.uint64)).all(), fmt_id(fmt)
        assert all(hgot[i] == dgot[i] for i in range(len(raws)) if hst[i] == A.OK), fmt_id(fmt)


def test_c2_shaped_gclz_and_chunklz10(codec):
    """4 096 files of 64 KiB from the C2 mix as GCLZ and as ChunkLZ10 with 4 KiB chunks: device equals host"""
    import torch
    from auroralib.compression_b200 import corpus
    dev = torch.device("cuda", 0)
    n, size = 4096, 65536
    raw, _ = corpus.generate_mix(n, size, device=dev)
    raw_h = raw.reshape(n, size).cpu().numpy()
    raws = [raw_h[i].tobytes() for i in range(n)]
    for fmt, opts in ((A.FMT_GCLZ, A.make_opts(quality=8)), (A.FMT_LZ77, A.make_opts(quality=8, lz77_type=0xF7, lz77_chunk_size=0x1000))):
        _, st, _ = _same_as_host(codec, fmt, raws, [codec.encode_bound(fmt, size)] * n, opts, "C2")
        assert (st == A.OK).sum() >= n // 2, fmt_id(fmt)


def test_second_device(codec, oracle):
    if codec.device_count < 2:
        pytest.skip("one device in the context")
    raws = _raws(5900)
    for fmt in (A.FMT_GCLZ, A.FMT_LZ77, A.FMT_ECD, A.FMT_LZ00, A.FMT_FCMP):
        for kw in _opt_sets(fmt):
            opts = A.make_opts(**({"quality": 8} | kw))
            _same_as_host(codec, fmt, raws, [roomy(len(r)) for r in raws], opts, f"device 1 {kw}", device=1)
