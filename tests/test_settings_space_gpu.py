"""The option values the other GPU tests leave at their defaults, on the B200 (the same ground on the lane emulation:
tests/test_settings_space_simt.py):

  * MaxWindowBits on every encoder, with both finders forced: the widened window and chain table of api.cu
    fill_encode_params, distances the formats' tokens truncate, chain tables that alias on long streams, and the scratch of
    the largest tables;
  * the LZSS property space the decoder accepts, its rejection boundary, and the encoders on the same sets;
  * the qualities no other GPU test runs (1, 7, 11, 13, 14) on every flag format.

Every answer is compared with the oracle: status and bytes for the encoders; status, out_len, consumed and bytes for the
decoders.  Where the oracle's stream does not round-trip (a token writer dropped distance bits) its decode is compared, not
asserted."""
import numpy as np
import pytest

from auroralib.compression_b200 import AuroraError, BatchCodec
from auroralib.compression_b200 import _abi as A
from tests import tokens as T
from tests.test_encode_gpu import ENC_FORMATS, PAR_FORMATS_WIDE
from tests.test_scan_decode_gpu import check as scan_check
from tests.test_settings_space_simt import FILLS, LZSS_SETS, MWB, far_repeats, lzss_decode_cases, lzss_id, lzss_raws
from tests.test_wrapped_device_gpu import _device_call, _device_inputs
from tests.test_wrapped_encode_device_gpu import device_encode, roomy
from tests.util import fmt_id, synth

pytestmark = pytest.mark.gpu

PAR, SERIAL = A.STRATEGY_PARALLEL_FINDER, A.STRATEGY_SERIAL_FINDER
BYTE_ENC = [A.FMT_LZ4, A.FMT_LZ4_LEGACY, A.FMT_LZ4_BLOCK, A.FMT_LZO, A.FMT_SNAPPY, A.FMT_SNAPPY_BLOCK, A.FMT_PRS]


def finders(fmt):
    return [0] if fmt in BYTE_ENC else [PAR, SERIAL]


def decode_both(codec, oracle, fmt, streams, caps, opts):
    """decode_batch and decode_device against the oracle: status, out_len, consumed, bytes"""
    import torch
    ref, rlen, rcons, rst = oracle.decode_batch(fmt, streams, caps, opts)
    outs, olen, cons, st = codec.decode_batch(fmt, streams, caps, opts)
    X = _device_inputs(streams, caps, torch.device("cuda", 0))
    torch.cuda.synchronize()
    _device_call(codec, fmt, X, opts)
    torch.cuda.synchronize()
    d_dst = X["d_dst"].cpu().numpy()
    d_st, d_olen, d_cons = X["d_st"].cpu().numpy(), X["d_olen"].cpu().numpy(), X["d_cons"].cpu().numpy()
    for what, s, o, c, got in (("host", st, olen, cons, lambda i: outs[i]),
                               ("device", d_st, d_olen, d_cons, lambda i: d_dst[int(X["doff"][i]):int(X["doff"][i]) + int(rlen[i])].tobytes())):
        bad = [i for i in range(len(streams)) if s[i] != rst[i] or int(o[i]) != int(rlen[i]) or int(c[i]) != int(rcons[i])
               or (rst[i] == 0 and got(i) != ref[i])]
        assert not bad, (f"{fmt_id(fmt)} {what}: {len(bad)}/{len(streams)} streams differ from the oracle; first #{bad[0]}: status "
                         f"{s[bad[0]]}/{rst[bad[0]]} out_len {o[bad[0]]}/{rlen[bad[0]]} consumed {c[bad[0]]}/{rcons[bad[0]]}")
    return rst


def encode_check(codec, oracle, fmt, raws, opts, what=""):
    got, st = codec.encode_batch(fmt, raws, opts)
    ref, rst = oracle.encode_batch(fmt, raws, opts)
    assert (st == rst).all(), (fmt_id(fmt), what, st, rst)
    bad = [i for i in range(len(raws)) if rst[i] == 0 and got[i] != ref[i]]
    assert not bad, f"{fmt_id(fmt)} {what}: {len(bad)}/{len(raws)} streams differ from the oracle; first #{bad[0]} len {len(raws[bad[0]])}"
    return ref, rst


def decode_what_does_not_round_trip(codec, oracle, fmt, raws, comps, rst):
    """the oracle's streams that its own decoder does not take back to the input: both decode entry points against its decode"""
    keep = [i for i in range(len(raws)) if rst[i] == 0 and len(raws[i])]
    if not keep:
        return 0
    streams, caps = [comps[i] for i in keep], [len(raws[i]) for i in keep]
    outs, _, _, st = oracle.decode_batch(fmt, streams, caps, A.make_opts())
    odd = [k for k in range(len(keep)) if not (st[k] == 0 and outs[k] == raws[keep[k]])]
    if odd:
        decode_both(codec, oracle, fmt, [streams[k] for k in odd], [caps[k] for k in odd], A.make_opts())
    return len(odd)


def mwb_raws(bmp, rng, quality):
    far = far_repeats(rng, bmp, 20000, [80000, 60000])   # copies 100 000 and 80 000 bytes apart
    raws = [bmp[:10], bmp[:10240], synth(rng, 4000, 0), synth(rng, 6000, 1), synth(rng, 5000, 2), synth(rng, 3000, 3)]
    if quality >= 13:   # (the sequential replay walks chains of 256+ candidates on one warp: short inputs)
        return raws + [far[:16000]]
    return raws + [far, bmp[:65536]]


@pytest.mark.parametrize("fmt", ENC_FORMATS, ids=fmt_id)
@pytest.mark.parametrize("quality", [1, 8, 15])
def test_max_window_bits(codec, oracle, bmp, fmt, quality):
    rng = np.random.default_rng(3100 + 16 * fmt + quality)
    raws = mwb_raws(bmp, rng, quality)
    odd = 0
    for mwb in MWB:
        # quality 1 and 28 bits: a 2^18-slot chain table, and a 300 KiB stream that reuses its slots
        longer = [bmp[:300 * 1024]] if quality == 1 and mwb == 28 else []
        for finder in finders(fmt):
            ref, rst = encode_check(codec, oracle, fmt, raws + longer, A.make_opts(quality=quality, max_window_bits=mwb, strategy=finder),
                                    f"q{quality} mwb {mwb} finder {finder:#x}")
        odd += decode_what_does_not_round_trip(codec, oracle, fmt, raws + longer, ref, rst)
    print(f"{fmt_id(fmt)} q{quality}: {odd} oracle streams that do not round-trip decoded on both entry points")


def test_max_window_bits_out_of_range(codec, bmp):
    import torch
    for mwb in (6, 29):
        for fmt in (A.FMT_LZ10, A.FMT_LZ4):
            opts = A.make_opts(quality=8, max_window_bits=mwb)
            with pytest.raises(AuroraError, match="INVALID_ARGUMENT"):
                codec.encode_batch(fmt, [bmp[:1000]], opts)
            with pytest.raises(AuroraError, match="INVALID_ARGUMENT"):
                device_encode(codec, fmt, [bmp[:1000]], [roomy(1000)], opts)
    torch.cuda.synchronize()


@pytest.mark.parametrize("fmt,kw", [(A.FMT_LZ10, {}), (A.FMT_LZ4, {}), (A.FMT_LZSS, {}), (A.FMT_GCLZ, {}), (A.FMT_LZ77, {"lz77_type": 0xF7})],
                         ids=["LZ10", "LZ4", "LZSS", "GCLZ", "LZ77-ChunkLZ10"])
def test_max_window_bits_device_and_wrappers(codec, oracle, bmp, fmt, kw):
    rng = np.random.default_rng(3300 + fmt)
    raws = [far_repeats(rng, bmp, 20000, [80000]), bmp[:70000], synth(rng, 5000, 2), bmp[:33]]
    for mwb in (16, 28):
        opts = A.make_opts(quality=8, max_window_bits=mwb, **kw)
        dgot, dst, dlen = device_encode(codec, fmt, raws, [roomy(len(r)) for r in raws], opts)
        hgot, hst = codec.encode_batch(fmt, raws, opts)
        for i, r in enumerate(raws):
            ref, rst = oracle.encode(fmt, r, opts)
            assert dst[i] == hst[i] == rst, (fmt_id(fmt), mwb, i, dst[i], hst[i], rst)
            assert dgot[i] == hgot[i] == ref, (fmt_id(fmt), mwb, i)


def test_scratch_of_the_widest_windows(oracle, bmp):
    """Quality 15 with MaxWindowBits 28: the largest hash (2^20) and chain (2^22 slots) tables.  One 64 KiB stream and a batch
    of 8 000 streams of 2 KiB, on a fresh context: the reference's bytes, not an allocation failure."""
    codec = BatchCodec(device_mask=1)
    try:
        opts = A.make_opts(quality=15, max_window_bits=28)
        many = [bmp[(i * 2048) % 900000:(i * 2048) % 900000 + 2048] for i in range(8000)]
        for fmt in (A.FMT_LZ10, A.FMT_LZ4):
            encode_check(codec, oracle, fmt, [bmp[:65536]], opts, "one 64 KiB stream")
            encode_check(codec, oracle, fmt, many, opts, "8000 x 2 KiB")
    finally:
        codec.close()


def test_the_lzss_sets_reach_both_decode_cores():
    from tests.test_settings_space_simt import test_the_sets_reach_both_decode_cores
    test_the_sets_reach_both_decode_cores()


@pytest.mark.parametrize("p", LZSS_SETS, ids=lzss_id)
def test_lzss_properties(codec, oracle, bmp, p):
    import torch
    lz = T.lzss_props(p)
    seed = 5100 + LZSS_SETS.index(p)
    streams, caps = lzss_decode_cases(oracle, p, seed, per_profile=6)
    for fill in FILLS:
        opts = A.make_opts(lzss=lz, lzss_initial_fill=fill)
        rst = decode_both(codec, oracle, A.FMT_LZSS, streams, caps, opts)
        assert (rst == 0).sum() >= len(streams) // 4
    # GetDecompressedSize on both entry points
    size, sst = codec.decoded_size_batch(A.FMT_LZSS, streams, A.make_opts(lzss=lz))
    X = _device_inputs(streams, caps, torch.device("cuda", 0))
    d_size = torch.full((len(streams),), -1, dtype=torch.int64, device="cuda")
    d_sst = torch.full((len(streams),), -9, dtype=torch.int32, device="cuda")
    codec.decoded_size_device(A.FMT_LZSS, X["d_src"], X["d_off"], X["d_len"], d_size, d_sst, A.make_opts(lzss=lz))
    torch.cuda.synchronize()
    for i, s in enumerate(streams):
        rs, rrst = oracle.decoded_size(A.FMT_LZSS, s, A.make_opts(lzss=lz))
        assert (int(size[i]), int(sst[i])) == (rs, rrst) or (sst[i] != 0 and rrst != 0), (lzss_id(p), i)
        assert int(d_size[i]) == int(size[i]) and int(d_sst[i]) == int(sst[i]), (lzss_id(p), i)
    # the offset scan over an image of the oracle's streams between junk
    rng = np.random.default_rng(seed)
    parts = []
    for x in lzss_raws(rng, bmp)[:4]:
        c, st = oracle.encode(A.FMT_LZSS, x, A.make_opts(quality=8, lzss=lz))
        assert st == 0
        parts += [c, rng.integers(0, 256, size=int(rng.integers(5, 60)), dtype=np.uint8).tobytes()]
    scan_check(codec, oracle, A.FMT_LZSS, b"".join(parts), A.make_opts(lzss=lz, lzss_initial_fill=FILLS[LZSS_SETS.index(p) % 3]))
    # the encoders on the same set
    raws = lzss_raws(rng, bmp)
    for q in (0, 8, 10):
        for finder in (PAR, SERIAL):
            encode_check(codec, oracle, A.FMT_LZSS, raws, A.make_opts(quality=q, lzss=lz, strategy=finder), f"{lzss_id(p)} q{q}")


def _hand_props(windows_bits=12, length_bits=8, min_length=255, max_distance=4096):
    lz = A.lz_props_bits(12, 8, 254)   # windows_bits 12, length_bits 8, max_distance 4096, min_length 255: every limit at once
    lz.windows_bits, lz.length_bits, lz.min_length, lz.max_distance = windows_bits, length_bits, min_length, max_distance
    return lz


@pytest.mark.parametrize("change", [{}, {"windows_bits": 13}, {"length_bits": 9}, {"max_distance": 4097}, {"min_length": 0},
                                    {"min_length": 256}], ids=["accepted", "wb13", "lb9", "dist4097", "min0", "min256"])
def test_lzss_rejection_boundary(codec, oracle, bmp, change):
    import torch
    accepted = _hand_props()
    lz = _hand_props(**change)
    rng = np.random.default_rng(5300)
    raws = lzss_raws(rng, bmp)
    comps, st = oracle.encode_batch(A.FMT_LZSS, raws, A.make_opts(quality=8, lzss=accepted))
    assert (st == 0).all()
    caps = [len(r) for r in raws]
    opts = A.make_opts(lzss=lz)
    image = b"".join(c + bytes(7) for c in comps)
    if not change:
        rst = decode_both(codec, oracle, A.FMT_LZSS, comps, caps, opts)
        assert (rst == 0).all()
        assert len(scan_check(codec, oracle, A.FMT_LZSS, image, opts)) == len(comps)
        return
    _, _, _, hst = codec.decode_batch(A.FMT_LZSS, comps, caps, opts)
    assert (hst == A.NOT_SUPPORTED).all(), hst
    # the device entry point rejects the whole call and launches nothing: the statuses keep what the caller put there
    X = _device_inputs(comps, caps, torch.device("cuda", 0))
    launches = codec.kernel_launches
    with pytest.raises(AuroraError, match="INVALID_ARGUMENT"):
        _device_call(codec, A.FMT_LZSS, X, opts)
    torch.cuda.synchronize()
    assert codec.kernel_launches == launches and (X["d_st"].cpu().numpy() == -9).all()
    d_img = torch.frombuffer(bytearray(image) + bytearray(16), dtype=torch.uint8).cuda()[:len(image)]
    s, *_ = codec.scan_decode_device(A.FMT_LZSS, d_img, opts)   # found 0 and the walk at the end, or it raises
    assert s.numel() == 0


@pytest.mark.parametrize("bad", [{"windows_bits": 25}, {"length_bits": 9}], ids=["wb25", "lb9"])
def test_lzss_encoder_rejects(codec, bmp, bad):
    opts = A.make_opts(quality=8, lzss=_hand_props(**bad))
    with pytest.raises(AuroraError, match="INVALID_ARGUMENT"):
        codec.encode_batch(A.FMT_LZSS, [bmp[:1000]], opts)
    with pytest.raises(AuroraError, match="INVALID_ARGUMENT"):
        device_encode(codec, A.FMT_LZSS, [bmp[:1000]], [roomy(1000)], opts)


@pytest.mark.parametrize("fmt", PAR_FORMATS_WIDE, ids=fmt_id)
@pytest.mark.parametrize("quality", [1, 7, 11, 13, 14])
def test_untested_qualities(codec, oracle, bmp, fmt, quality):
    rng = np.random.default_rng(3500 + 16 * fmt + quality)
    small = [bmp[:16000], synth(rng, 9000, 0), synth(rng, 7000, 1), synth(rng, 5000, 2), synth(rng, 3000, 3), bmp[:33]]
    for finder in (0, PAR, SERIAL):
        raws = small + ([] if quality >= 13 and finder != PAR else [bmp[:70000]])
        encode_check(codec, oracle, fmt, raws, A.make_opts(quality=quality, strategy=finder), f"q{quality} finder {finder:#x}")
