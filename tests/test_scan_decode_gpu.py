"""aurora_scan_decode_device (BatchCodec.scan_decode_device): the CLI's `-scan` walk on a device image, against the walk written
in Python — the bitmap of codec.scan_offsets (pinned to the oracle by test_ismatch_gpu.py) and the oracle's decode of every
visited hit at capacity max_size, so no GPU call runs inside the reference."""
import ctypes as C

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests.util import corrupt, fmt_id, rom_like_image, synth

pytestmark = pytest.mark.gpu

SCAN_FORMATS = [A.FMT_YAZ0, A.FMT_YAZ1, A.FMT_YAY0, A.FMT_MIO0, A.FMT_LZ10, A.FMT_LZ11, A.FMT_LZSS, A.FMT_LZ4, A.FMT_LZ4_LEGACY,
                A.FMT_LZO, A.FMT_SNAPPY, A.FMT_PRS, A.FMT_LZHUDSON, A.FMT_LZ40, A.FMT_LZ60, A.FMT_SMSR00]
REFUSED = [A.FMT_LZ4_BLOCK, A.FMT_SNAPPY_BLOCK, A.FMT_BLZ, A.FMT_GCLZ, A.FMT_LZ77, A.FMT_LEVEL5, A.FMT_LZ00, A.FMT_ECD, 0, 99]
MAX = 1 << 14


def ref_walk(codec, oracle, fmt, image, opts=None, max_size=MAX, begin=0):
    """-> list of (start, consumed, out_len, bytes): the walk of the header, decodes from the oracle in chunks of hits."""
    bitmap = codec.scan_offsets(fmt, image, opts) if len(image) else np.zeros(0, dtype=bool)
    hits = [int(h) for h in np.nonzero(bitmap)[0] if h >= begin]
    index = {h: k for k, h in enumerate(hits)}
    base = np.frombuffer(image, dtype=np.uint8).copy() if len(image) else np.zeros(16, dtype=np.uint8)
    res = {}

    def outcome(h):
        if h not in res:
            k = index[h]
            chunk = hits[k:k + 1024]
            off = np.array(chunk, dtype=np.uint64)
            ln = np.uint64(len(image)) - off
            caps = np.full(len(chunk), max_size, dtype=np.uint64)
            doff = np.arange(len(chunk), dtype=np.uint64) * np.uint64((max_size + 15) & ~15)
            dst = np.zeros(len(chunk) * ((max_size + 15) & ~15) + 16, dtype=np.uint8)
            out_len, consumed, status = oracle.decode_packed(fmt, base, off, ln, dst, doff, caps, opts)
            for j, c in enumerate(chunk):
                ol = int(out_len[j])
                res[c] = (int(status[j]), int(consumed[j]), ol, dst[int(doff[j]):int(doff[j]) + min(ol, max_size)].tobytes())
        return res[h]

    hitset, entries, i = set(hits), [], begin
    while i < len(image):
        if i in hitset:
            st, c, ol, data = outcome(i)
            if st == A.OK:
                entries.append((i, c, ol, data))
                i += max(c, 1)
                continue
        i += 1
    return entries


def device_walk(codec, fmt, image, opts=None, max_size=MAX, begin=0):
    import torch
    d_img = torch.frombuffer(bytearray(image) + bytearray(16), dtype=torch.uint8).cuda()[:len(image)]
    before = d_img.clone()
    s, c, ol, dst, off = codec.scan_decode_device(fmt, d_img, opts, max_size=max_size, begin=begin)
    torch.cuda.synchronize()
    assert torch.equal(d_img, before)
    s, c, ol, off = (x.cpu().tolist() for x in (s, c, ol, off))
    dst = dst.cpu().numpy().tobytes()
    want_off, pos = [], 0
    for n in ol:
        want_off.append(pos)
        pos += (n + 15) & ~15
    assert off == want_off
    return [(s[k], c[k], ol[k], dst[off[k]:off[k] + ol[k]]) for k in range(len(s))]


def check(codec, oracle, fmt, image, opts=None, max_size=MAX, begin=0, min_entries=0):
    want = ref_walk(codec, oracle, fmt, image, opts, max_size, begin)
    got = device_walk(codec, fmt, image, opts, max_size, begin)
    assert [e[:3] for e in got] == [e[:3] for e in want], fmt_id(fmt)
    for g, w in zip(got, want):
        assert g[3] == w[3], (fmt_id(fmt), g[0])
    assert len(got) >= min_entries, (fmt_id(fmt), len(got))
    return got


def assets(rng, bmp):
    return [bmp[1000:9000], bytes(3000), synth(rng, 5000, 0), synth(rng, 2500, 2)]


@pytest.mark.parametrize("fmt", SCAN_FORMATS, ids=fmt_id)
def test_rom_like_images_and_edge_images(codec, oracle, bmp, fmt):
    rng = np.random.default_rng(4100 + fmt)
    a = assets(rng, bmp)
    image, starts = rom_like_image(oracle, rng, fmt, a)
    got = check(codec, oracle, fmt, image)
    if fmt in (A.FMT_YAZ0, A.FMT_YAZ1, A.FMT_MIO0, A.FMT_LZ4, A.FMT_LZSS, A.FMT_SMSR00):   # magic formats find every asset
        assert [e[3] for e in got if e[0] in starts] == a
    # back to back, no junk
    comp = [oracle.encode(fmt, x, A.make_opts(quality=8))[0] for x in a]
    check(codec, oracle, fmt, b"".join(comp))
    # a flipped byte and a truncated asset: the walk steps by one and meets hits inside the broken stream
    broken = corrupt(rng, comp[0], 1) + comp[1][:len(comp[1]) // 2] + comp[2] + comp[3]
    check(codec, oracle, fmt, broken)
    # an asset larger than max_size, then one that fits
    check(codec, oracle, fmt, comp[0] + comp[3], max_size=4000)
    # no hits; 0, 1 and 15 bytes
    for img in (bytes(5000), b"", b"\x10", image[:15], comp[3][:15]):
        check(codec, oracle, fmt, img)


@pytest.mark.parametrize("fmt", [A.FMT_YAZ0, A.FMT_YAZ1, A.FMT_MIO0], ids=fmt_id)
def test_little_endian_assets_under_the_default_order(codec, oracle, bmp, fmt):
    rng = np.random.default_rng(4200 + fmt)
    parts = []
    for x in assets(rng, bmp):
        c, st = oracle.encode(fmt, x, A.make_opts(quality=8, byte_order=A.ENDIAN_LITTLE))
        assert st == 0
        parts += [c, rng.integers(0, 256, size=50, dtype=np.uint8).tobytes()]
    image = b"".join(parts)
    for opts in (None, A.make_opts(byte_order=A.ENDIAN_LITTLE), A.make_opts(byte_order=A.ENDIAN_BIG)):
        check(codec, oracle, fmt, image, opts, max_size=MAX)
    got = check(codec, oracle, fmt, image, None, max_size=MAX, min_entries=1)
    assert got[0][0] == 0


def test_lz4_content_checksums_under_lz4_verify(codec, oracle, bmp):
    rng = np.random.default_rng(4300)
    parts, raws = [], []
    for k, x in enumerate(assets(rng, bmp)):
        c, st = oracle.encode(A.FMT_LZ4, x, A.make_opts(quality=8))
        frame = bytearray(c)
        frame[4] |= 0x04   # content checksum present
        sum_ = oracle.xxh32(x) ^ (0x5A if k % 2 else 0)   # odd assets carry a wrong checksum
        parts += [bytes(frame) + sum_.to_bytes(4, "little"), rng.integers(0, 256, size=40, dtype=np.uint8).tobytes()]
    image = b"".join(parts)
    verified = check(codec, oracle, A.FMT_LZ4, image, A.make_opts(lz4_verify=1))
    unverified = check(codec, oracle, A.FMT_LZ4, image, A.make_opts(lz4_verify=0))
    assert len(verified) < len(unverified)


def test_lzss_with_other_properties(codec, oracle, bmp):
    rng = np.random.default_rng(4400)
    props = A.LzProps()
    codec._L.aurora_lz_props_bits(C.byref(props), 10, 6, 2)
    opts = A.make_opts(quality=8, lzss=props)
    parts = []
    for x in assets(rng, bmp):
        c, st = oracle.encode(A.FMT_LZSS, x, opts)
        assert st == 0
        parts += [c, rng.integers(0, 256, size=30, dtype=np.uint8).tobytes()]
    got = check(codec, oracle, A.FMT_LZSS, b"".join(parts), A.make_opts(lzss=props))
    assert len(got) == 4


def prs_stream_image(oracle, rng, count):
    """`count` tiny PRS streams (a pool of 64 that pass PRS's IsMatch) with 0-3 junk bytes after each: PRS's token walk
    rarely accepts random bytes, so a PRS image with more hits than one round keeps is made of real streams."""
    pool = []
    while len(pool) < 64:
        c, st = oracle.encode(A.FMT_PRS, bytes(rng.integers(0, 4, size=int(rng.integers(6, 24)), dtype=np.uint8)),
                              A.make_opts(quality=8))
        if st == 0 and oracle.is_match(A.FMT_PRS, c + bytes(8)):
            pool.append(c)
    picks = rng.integers(0, len(pool), size=count)
    gaps = rng.integers(0, 4, size=count)
    return b"".join(pool[p] + rng.integers(0, 256, size=int(g), dtype=np.uint8).tobytes() for p, g in zip(picks, gaps))


@pytest.mark.parametrize("fmt", [A.FMT_LZO, A.FMT_PRS], ids=fmt_id)
def test_hits_that_span_several_rounds(codec, oracle, fmt):
    rng = np.random.default_rng(4500 + fmt)
    if fmt == A.FMT_LZO:   # random junk: every byte below 0x20 is an LZO hit
        image = rng.integers(0, 256, size=640 << 10, dtype=np.uint8).tobytes()
    else:
        image = prs_stream_image(oracle, rng, 70000)
    assert int(codec.scan_offsets(fmt, image).sum()) > (1 << 16)   # more hits than one round keeps
    got = check(codec, oracle, fmt, image, max_size=1024)
    if fmt == A.FMT_PRS:
        assert len(got) > (1 << 16)


def test_resumption_and_pieces(codec, oracle, bmp):
    import torch
    rng = np.random.default_rng(4600)
    fmt = A.FMT_YAZ0
    image, starts = rom_like_image(oracle, rng, fmt, assets(rng, bmp) * 3)
    full = ref_walk(codec, oracle, fmt, image)
    for b in [0, 1, starts[2], starts[2] + 1, starts[5] - 3, len(image) - 1, len(image)]:
        assert [e[:3] for e in device_walk(codec, fmt, image, begin=b)] == [e[:3] for e in full if e[0] >= b]
    d_img = torch.frombuffer(bytearray(image), dtype=torch.uint8).cuda()
    L, ctx = codec._L, codec._ctx
    opts = A.make_opts()

    def piece(pos, max_found, dst_bytes, sentinel=0xA5):
        d = [torch.full((64,), -7, dtype=torch.int64, device="cuda") for _ in range(4)]
        dst = torch.full((dst_bytes + 64,), sentinel, dtype=torch.uint8, device="cuda")
        found, nxt = C.c_uint64(), C.c_uint64()
        torch.cuda.synchronize()   # the sentinels are written on torch's stream, the call runs on the library's
        rc = L.aurora_scan_decode_device(ctx, 0, fmt, C.byref(opts), d_img.data_ptr(), len(image), pos, MAX, max_found, d[0].data_ptr(),
                                         d[1].data_ptr(), d[2].data_ptr(), dst.data_ptr(), dst_bytes, d[3].data_ptr(), C.byref(found),
                                         C.byref(nxt), None)
        assert rc == A.OK
        k = found.value
        for x in d:
            assert (x[k:] == -7).all()   # descriptors past *found untouched
        hd = dst.cpu().numpy()
        mask = np.ones(len(hd), dtype=bool)
        ents = []
        for j in range(k):
            o, n = int(d[3][j]), int(d[2][j])
            mask[o:o + n] = False
            ents.append((int(d[0][j]), int(d[1][j]), n, hd[o:o + n].tobytes()))
        assert (hd[mask] == sentinel).all()   # nothing outside the entries' bytes
        return ents, nxt.value

    for max_found in (1, 2):
        got, pos = [], 0
        while pos < len(image):
            ents, pos = piece(pos, max_found, 1 << 20)
            got += ents
        assert got == full
    # a destination one byte short of entry 1's end stops before entry 1
    end1 = ((full[0][2] + 15) & ~15) + full[1][2]
    ents, nxt = piece(0, 64, end1 - 1)
    assert [e[:3] for e in ents] == [full[0][:3]] and nxt == full[1][0]
    ents, nxt = piece(nxt, 64, 1 << 20)
    assert ents == full[1:] and nxt == len(image)


def test_rejections_launch_nothing(codec):
    import torch
    L, ctx = codec._L, codec._ctx
    img = torch.zeros(4096 + 16, dtype=torch.uint8, device="cuda")
    d = [torch.zeros(8, dtype=torch.int64, device="cuda") for _ in range(4)]
    dst = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    found, nxt = C.c_uint64(99), C.c_uint64(99)

    def call(fmt, ptr=img.data_ptr(), length=4096, begin=0, max_size=MAX):
        return L.aurora_scan_decode_device(ctx, 0, fmt, C.byref(A.make_opts()), ptr, length, begin, max_size, 8, d[0].data_ptr(),
                                           d[1].data_ptr(), d[2].data_ptr(), dst.data_ptr(), 4096, d[3].data_ptr(), C.byref(found),
                                           C.byref(nxt), None)
    before = codec.kernel_launches
    for fmt in REFUSED:
        assert call(fmt) == A.INVALID_ARGUMENT, fmt
    assert b"aurora_scan_offsets" in L.aurora_last_error_string(ctx)
    assert call(A.FMT_YAZ0, ptr=img.data_ptr() + 1) == A.INVALID_ARGUMENT
    assert call(A.FMT_YAZ0, begin=4097) == A.INVALID_ARGUMENT
    assert call(A.FMT_YAZ0, max_size=0) == A.INVALID_ARGUMENT
    assert call(A.FMT_YAZ0, max_size=1 << 32) == A.INVALID_ARGUMENT
    assert call(A.FMT_YAZ0, ptr=0) == A.INVALID_ARGUMENT
    for length, begin in ((0, 0), (4096, 4096)):
        assert call(A.FMT_YAZ0, length=length, begin=begin) == A.OK and (found.value, nxt.value) == (0, length)
    assert codec.kernel_launches == before


def test_non_default_stream_behind_busy_work(codec, oracle, bmp):
    import torch
    rng = np.random.default_rng(4700)
    image, starts = rom_like_image(oracle, rng, A.FMT_LZ4, assets(rng, bmp))
    want = ref_walk(codec, oracle, A.FMT_LZ4, image)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        d_img = torch.frombuffer(bytearray(image), dtype=torch.uint8).cuda()
        x = torch.randn(4096, 4096, device="cuda")
        for _ in range(8):
            x = x @ x / 64
        got = codec.scan_decode_device(A.FMT_LZ4, d_img, max_size=MAX, stream=s.cuda_stream)
    torch.cuda.synchronize()
    st, c, ol, dst, off = (t.cpu() for t in got)
    assert st.tolist() == [e[0] for e in want] and ol.tolist() == [e[2] for e in want]
    assert [dst[o:o + n].numpy().tobytes() for o, n in zip(off.tolist(), ol.tolist())] == [e[3] for e in want]


@pytest.mark.parametrize("fmt", [A.FMT_YAZ0, A.FMT_LZ4], ids=fmt_id)
def test_scale_4096_c2_assets(codec, fmt):
    import torch
    from auroralib.compression_b200.corpus import generate_mix
    raw, _ = generate_mix(4096, 8192)
    raw = raw.numpy()
    blobs = [raw[i].tobytes() for i in range(len(raw))]
    comp, status = codec.encode_batch(fmt, blobs, A.make_opts(quality=8))
    assert (status == 0).all()
    rng = np.random.default_rng(4800)
    parts, starts, pos = [], [], 0
    for c in comp:
        j = rng.integers(0, 256, size=int(rng.integers(1, 200)), dtype=np.uint8).tobytes()
        parts += [j, c]
        starts.append(pos + len(j))
        pos += len(j) + len(c)
    image = b"".join(parts)
    d_img = torch.frombuffer(bytearray(image), dtype=torch.uint8).cuda()
    st, c, ol, dst, off = (t.cpu() for t in codec.scan_decode_device(fmt, d_img, max_size=1 << 16))
    assert st.tolist() == starts and c.tolist() == [len(x) for x in comp]
    dst = dst.numpy()
    assert all(dst[o:o + 8192].tobytes() == b for o, b in zip(off.tolist(), blobs))


def test_second_device(codec, oracle, bmp):
    import torch
    if codec.device_count < 2 or torch.cuda.device_count() < 2:
        pytest.skip("one device")
    rng = np.random.default_rng(4900)
    image, starts = rom_like_image(oracle, rng, A.FMT_MIO0, assets(rng, bmp))
    want = ref_walk(codec, oracle, A.FMT_MIO0, image)
    with torch.cuda.device(1):
        d_img = torch.frombuffer(bytearray(image), dtype=torch.uint8).to("cuda:1")
        st, c, ol, dst, off = (t.cpu() for t in codec.scan_decode_device(A.FMT_MIO0, d_img, max_size=MAX, device=1))
    assert st.tolist() == [e[0] for e in want] and c.tolist() == [e[1] for e in want]
    assert [dst[o:o + n].numpy().tobytes() for o, n in zip(off.tolist(), ol.tolist())] == [e[3] for e in want]
