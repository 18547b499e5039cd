"""GPU tests of batches whose source windows share bytes: one window listed several times, a window and its extensions (encode:
prefixes of one buffer), windows that start inside one another, and the scan chain of an image (every file start to the end
of the image, so every window contains the ones after it), each also in descending offset order.  Every pattern runs in a
dense source, which the host entry points copy to the device as one span, and in a sparse one (two copies of the pattern
more than 1.25 x their summed length + 1 MiB apart), which they re-lay out stream by stream.

Every result equals that of the same window processed alone: decode (host and device entry points) the status, out_len,
consumed and destination bytes of a one-stream host batch, which equal the oracle's; encode the oracle's bytes, and the device
entry point the host's; the queries the per-window answer.  No call changes its source.  LZ00's keystream and BLZ's reversal
rewrite a device copy of the source in place, so these batches are where a copy shared by two windows would show."""
import numpy as np
import pytest

from auroralib.compression_b200 import layout
from auroralib.compression_b200 import _abi as A
from tests.test_encode_gpu import ENC_FORMATS
from tests.test_wrapped_encode_device_gpu import _oracle_ref
from tests.test_wrappers import _opt_sets
from tests.util import ALL_FORMATS, MATCHABLE, SIZED_FORMATS, fmt_id, synth

pytestmark = pytest.mark.gpu

WRAPPERS = A.WRAPPER_FORMATS
BYTELZ = [A.FMT_LZ4, A.FMT_LZ4_BLOCK, A.FMT_LZ4_LEGACY, A.FMT_LZO, A.FMT_SNAPPY, A.FMT_SNAPPY_BLOCK, A.FMT_PRS]
NO_SCAN = (A.FMT_LZ4_BLOCK, A.FMT_SNAPPY_BLOCK, A.FMT_BLZ)   # formats without an offset scan: the known file starts
PATTERNS = ["repeat", "nest", "overlap", "scan_chain"]
SENTINEL = 0x5A
NO_IS_MATCH = (A.FMT_LEVEL5, A.FMT_LZSEGA, A.FMT_GCZ)   # wrappers whose IsMatch needs zlib or the file name: NOT_SUPPORTED


def a16(v):
    return (int(v) + 15) & ~15


def opts_of(fmt, kw):
    return A.make_opts(**({"quality": 8} | kw))


# ------------------------------------------------------------------------------------------------------------ the batches
def place(blobs):
    """blobs back to back at 16-byte aligned offsets -> (image bytes, start of every blob); the image ends with the last blob"""
    image, starts = bytearray(), []
    for b in blobs:
        image += bytes(a16(len(image)) - len(image))
        starts.append(len(image))
        image += b
    return bytes(image), starts


def windows(pattern, image, starts, lens, chain):
    """(offset, length) windows of one pattern over an image whose blobs 0, 1, ... are at starts with lengths lens; the last
    blob is an unrelated stream.  chain: the window starts of the scan chain (each window runs to the end of the image)."""
    E = len(image)
    s0, l0, s1, l1, su, lu = starts[0], lens[0], starts[1], lens[1], starts[-1], lens[-1]
    if pattern == "repeat":
        return [(s0, l0), (su, lu), (s0, l0), (s1, l1), (s0, l0)]
    if pattern == "nest":   # a window, the same window extended by trailing bytes, and the rest of the image
        return [(s0, l0), (s0, min(l0 + 53, E - s0)), (s0, l0 + 1), (s0, E - s0)]
    if pattern == "overlap":   # windows that start inside one another at different offsets
        step = max(16, (l0 // 3) & ~15)
        return [(s0 + j * step, min(l0 + 16 * j + 40, E - s0 - j * step)) for j in range(4)] + [(s1 - 16, min(l1, E - s1 + 16))]
    assert pattern == "scan_chain"
    return [(s, E - s) for s in chain]


def layouts(image, wins):
    """dense: the pattern over the image itself; sparse: the pattern over two copies of the image placed so far apart that the
    windows' extent exceeds 1.25 x their summed length + 1 MiB + 64 per stream (the host entry points' packed layout)"""
    total = 2 * sum(l for _, l in wins)
    gap = a16(len(image) + total + total // 4 + (1 << 20) + 64 * 2 * len(wins) + 4096)
    sparse = np.zeros(gap + a16(len(image)) + 16, dtype=np.uint8)
    sparse[:len(image)] = np.frombuffer(image, dtype=np.uint8)
    sparse[gap:gap + len(image)] = np.frombuffer(image, dtype=np.uint8)
    dense = np.zeros(a16(len(image)) + 16, dtype=np.uint8)
    dense[:len(image)] = np.frombuffer(image, dtype=np.uint8)
    return [("dense", dense, wins, 0), ("sparse", sparse, wins + [(o + gap, l) for o, l in wins], gap)]


def variants(image, wins, with_image_offsets=False):
    """every (layout, order) of a pattern -> (name, source array, offsets u64, lengths u64[, every window's offset in the image])"""
    for order in ("ascending", "descending"):
        w = wins if order == "ascending" else sorted(wins, key=lambda x: -x[0])
        for lay, src, ww, gap in layouts(image, w):
            r = (f"{lay} {order}", src, np.array([o for o, _ in ww], dtype=np.uint64), np.array([l for _, l in ww], dtype=np.uint64))
            yield r + ([o if o < gap or not gap else o - gap for o, _ in ww],) if with_image_offsets else r


def t64(dev, a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).astype(np.int64)).to(dev)


def device_source(dev, src):
    import torch
    return torch.from_numpy(src.copy()).to(dev)


# ------------------------------------------------------------------------------------------------------------ decode
class Alone:
    """the answers of one window processed alone (a one-stream host batch), cached by its bytes and capacity"""

    def __init__(self, codec, oracle, fmt, opts):
        self.codec, self.oracle, self.fmt, self.opts, self.memo = codec, oracle, fmt, opts, {}

    def decode(self, blob, cap):
        k = (blob, cap)
        if k not in self.memo:
            outs, olen, cons, st = self.codec.decode_batch(self.fmt, [blob], [cap], self.opts)
            r_outs, r_olen, r_cons, r_st = self.oracle.decode_batch(self.fmt, [blob], [cap], self.opts)
            assert (st[0], olen[0], cons[0]) == (r_st[0], r_olen[0], r_cons[0]) and outs[0] == r_outs[0], \
                f"{fmt_id(self.fmt)}: a one-stream batch differs from the oracle ({st[0]}/{r_st[0]}, {olen[0]}/{r_olen[0]})"
            self.memo[k] = (int(st[0]), int(olen[0]), int(cons[0]), outs[0])
        return self.memo[k]


def compare_decode(fmt, what, alone, src, off, ln, caps, doff, dst, olen, cons, st):
    for i in range(len(off)):
        blob = src[int(off[i]):int(off[i]) + int(ln[i])].tobytes()
        a_st, a_olen, a_cons, a_out = alone.decode(blob, int(caps[i]))
        got = dst[int(doff[i]):int(doff[i]) + min(int(olen[i]), int(caps[i]))].tobytes()
        assert (int(st[i]), int(olen[i]), int(cons[i])) == (a_st, a_olen, a_cons) and got == a_out, (
            f"{fmt_id(fmt)} {what}: window #{i} at {int(off[i])} (+{int(ln[i])}): status {st[i]} / alone {a_st}, out_len "
            f"{olen[i]} / {a_olen}, consumed {cons[i]} / {a_cons}, bytes {'equal' if got == a_out else 'differ'}")


def decode_both(codec, fmt, opts, what, alone, src, off, ln, caps):
    """the host and the device entry point on one batch, each against the windows alone; -> host (out_len, status, windows)"""
    import torch
    caps, doff, total = layout(caps)
    before = src.copy()
    h_dst = np.full(total + 64, SENTINEL, dtype=np.uint8)
    olen, cons, st = codec.decode_packed(fmt, src, off, ln, h_dst, doff, caps, opts)
    assert np.array_equal(src, before), f"{fmt_id(fmt)} {what}: the host source changed"
    compare_decode(fmt, what + " (host)", alone, src, off, ln, caps, doff, h_dst, olen, cons, st)

    dev = torch.device("cuda", 0)
    d_src = device_source(dev, src)
    n = len(off)
    d_dst = torch.full((total + 64,), SENTINEL, dtype=torch.uint8, device=dev)
    d_olen = torch.full((n,), -1, dtype=torch.int64, device=dev)
    d_cons = torch.full((n,), -1, dtype=torch.int64, device=dev)
    d_st = torch.full((n,), -9, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    codec.decode_device(fmt, d_src, t64(dev, off), t64(dev, ln), d_dst, t64(dev, doff), t64(dev, caps), d_olen, d_cons, d_st, opts)
    torch.cuda.synchronize(dev)
    assert np.array_equal(d_src.cpu().numpy(), before), f"{fmt_id(fmt)} {what}: the device source changed"
    compare_decode(fmt, what + " (device)", alone, src, off, ln, caps, doff, d_dst.cpu().numpy(), d_olen.cpu().numpy().astype(np.uint64),
                   d_cons.cpu().numpy().astype(np.uint64), d_st.cpu().numpy())
    return olen, st, [h_dst[int(doff[i]):int(doff[i]) + min(int(olen[i]), int(caps[i]))].tobytes() for i in range(n)]


def decode_files(oracle, fmt, opts, seed):
    """three files of several KiB and an unrelated stream, encoded by the oracle -> (raws, comps)"""
    rng = np.random.default_rng(seed)
    raws = [synth(rng, n, k) for n, k in ((9000, 0), (6000, 2), (12000, 1), (3000, 3))]
    comps = []
    for r in raws:
        c, st = oracle.encode(fmt, r, opts)
        assert st == 0, (fmt_id(fmt), st)
        comps.append(c)
    return raws, comps


def chain_starts(codec, fmt, opts, image, starts):
    """the scan chain's window starts: the 16-byte aligned hits of the offset scan (at most 12 besides the files) and the files"""
    if fmt in NO_SCAN or fmt in WRAPPERS:
        return list(starts)
    hits = [int(h) for h in np.nonzero(codec.scan_offsets(fmt, image, opts))[0] if h % 16 == 0 and h not in starts]
    return sorted(set(starts) | set(hits[:12]))


@pytest.mark.parametrize("pattern", PATTERNS)
@pytest.mark.parametrize("fmt", ALL_FORMATS + WRAPPERS, ids=fmt_id)
def test_decode(codec, oracle, fmt, pattern):
    for kw in _opt_sets(fmt) if fmt in WRAPPERS else [dict()]:
        opts = opts_of(fmt, kw)
        raws, comps = decode_files(oracle, fmt, opts, 4100 + fmt)
        alone = Alone(codec, oracle, fmt, opts)
        files = comps[:3] if pattern == "scan_chain" else comps
        image, starts = place(files)
        chain = chain_starts(codec, fmt, opts, image, starts) if pattern == "scan_chain" else []
        wins = windows(pattern, image, starts, [len(c) for c in files], chain)
        cap = max(len(r) for r in raws) + 64
        for name, src, off, ln, at in variants(image, wins, with_image_offsets=True):
            what = f"{pattern} {name} {kw}"
            olen, st, outs = decode_both(codec, fmt, opts, what, alone, src, off, ln, [cap] * len(off))
            if pattern != "scan_chain":
                continue
            # the files of the chain decode to their raw bytes (BLZ reads from the end of its window: the last file)
            for i in range(len(off)):
                if at[i] not in starts:
                    continue
                k = starts.index(at[i])
                if fmt == A.FMT_BLZ:
                    k = len(files) - 1
                if fmt in (A.FMT_LZON, A.FMT_SDPC) and outs[i] != raws[k]:
                    continue   # the LZO encoder's dropped-first-match quirk (DESIGN.md section 2)
                if fmt == A.FMT_SNAPPY and at[i] != starts[-1]:
                    continue   # (a framed Snappy stream reads on through the frames of the files behind it)
                if st[i] == A.OK or at[i] == starts[-1] or fmt == A.FMT_LZ00:
                    assert st[i] == A.OK and outs[i] == raws[k], f"{fmt_id(fmt)} {what}: chain file {k} (window #{i}): status {st[i]}"


# ------------------------------------------------------------------------------------------------------------ encode
def encode_bound(codec, fmt, n):
    return max(codec.encode_bound(fmt, n), 8 + 2 * (n + 2) + 3 * n + 70 * (n // 0x400 + 2) + 1024)


def encode_both(codec, oracle, fmt, kw, opts, what, memo, src, off, ln):
    import torch
    caps, doff, total = layout([encode_bound(codec, fmt, int(x)) for x in ln])
    before = src.copy()
    h_dst = np.full(total + 64, SENTINEL, dtype=np.uint8)
    olen, st = codec.encode_packed(fmt, src, off, ln, h_dst, doff, caps, opts)
    assert np.array_equal(src, before), f"{fmt_id(fmt)} {what}: the host source changed"
    for i in range(len(off)):
        raw = src[int(off[i]):int(off[i]) + int(ln[i])].tobytes()
        if raw not in memo:
            memo[raw] = _oracle_ref(oracle, fmt, raw, kw, opts)
        ref, rst = memo[raw]
        got = h_dst[int(doff[i]):int(doff[i]) + int(olen[i])].tobytes() if st[i] == A.OK else None
        assert st[i] == rst and (st[i] != A.OK or got == ref), (
            f"{fmt_id(fmt)} {what}: window #{i} at {int(off[i])} (+{int(ln[i])}): status {st[i]} / oracle {rst}, "
            f"{olen[i]} / {len(ref)} bytes, {'equal' if got == ref else 'differ'}")
    if fmt == A.FMT_BLZ:
        return   # (BLZ encodes on the host entry point only)
    dev = torch.device("cuda", 0)
    d_src = device_source(dev, src)
    n = len(off)
    d_dst = torch.full((total + 64,), SENTINEL, dtype=torch.uint8, device=dev)
    d_olen = torch.full((n,), -1, dtype=torch.int64, device=dev)
    d_st = torch.full((n,), -9, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    codec.encode_device(fmt, d_src, t64(dev, off), t64(dev, ln), d_dst, t64(dev, doff), t64(dev, caps), d_olen, d_st, opts)
    torch.cuda.synchronize(dev)
    assert np.array_equal(d_src.cpu().numpy(), before), f"{fmt_id(fmt)} {what}: the device source changed"
    g_dst, g_olen, g_st = d_dst.cpu().numpy(), d_olen.cpu().numpy(), d_st.cpu().numpy()
    for i in range(n):
        m = min(int(olen[i]), int(caps[i]))
        same = g_dst[int(doff[i]):int(doff[i]) + m].tobytes() == h_dst[int(doff[i]):int(doff[i]) + m].tobytes()
        assert g_st[i] == st[i] and g_olen[i] == int(olen[i]) and (st[i] != A.OK or same), (
            f"{fmt_id(fmt)} {what} (device): window #{i}: status {g_st[i]} / host {st[i]}, out_len {g_olen[i]} / {olen[i]}")


@pytest.mark.parametrize("pattern", PATTERNS)
@pytest.mark.parametrize("fmt", ENC_FORMATS + WRAPPERS, ids=fmt_id)
def test_encode(codec, oracle, fmt, pattern):
    rng = np.random.default_rng(4200 + fmt)
    buf, other = synth(rng, 12000, 2), synth(rng, 3000, 0)
    image, starts = place([buf, other])
    E = len(buf)
    if pattern == "nest":   # several prefixes of one buffer, lengths 1 and 0 included
        wins = [(0, E), (0, E // 2), (0, 1), (0, 0), (0, E - 1), (0, 4097)]
    elif pattern == "scan_chain":   # suffixes: every window runs to the end of the image
        wins = [(s, len(image) - s) for s in (0, 16 * 97, 16 * 300, 16 * 601, starts[1])]
    else:
        wins = windows(pattern, image, starts + [starts[1]], [E, len(other), len(other)], [])
    for kw in _opt_sets(fmt) if fmt in WRAPPERS else [dict()]:
        opts = opts_of(fmt, kw)
        memo = {}
        for name, src, off, ln in variants(image, wins):
            encode_both(codec, oracle, fmt, kw, opts, f"{pattern} {name} {kw}", memo, src, off, ln)


# ------------------------------------------------------------------------------------------------------------ queries
@pytest.mark.parametrize("fmt", ALL_FORMATS + WRAPPERS, ids=fmt_id)
def test_queries(codec, oracle, fmt):
    import torch
    dev = torch.device("cuda", 0)
    opts = opts_of(fmt, _opt_sets(fmt)[-1] if fmt in WRAPPERS else dict())
    raws, comps = decode_files(oracle, fmt, opts, 4300 + fmt)
    image, starts = place(comps)
    scan = fmt in BYTELZ
    match_fmt = fmt in MATCHABLE or (fmt in WRAPPERS and fmt not in NO_IS_MATCH)
    size_fmt = fmt in SIZED_FORMATS or scan or fmt in WRAPPERS
    memo_m, memo_s = {}, {}
    for pattern in PATTERNS:
        wins = windows(pattern, image, starts, [len(c) for c in comps], starts)
        for name, src, off, ln in variants(image, wins):
            what = f"{pattern} {name}"
            before = src.copy()
            blobs = [src[int(o):int(o) + int(l)].tobytes() for o, l in zip(off, ln)]
            d_src = device_source(dev, src)
            d_off, d_len = t64(dev, off), t64(dev, ln)
            n = len(off)
            if match_fmt:
                m = codec.is_match_packed(fmt, src, off, ln, opts)
                want = np.array([memo_m.setdefault(b, bool(codec.is_match_batch(fmt, [b], opts)[0])) for b in blobs])
                assert np.array_equal(m, want), f"{fmt_id(fmt)} {what}: IsMatch {m.astype(int)} / alone {want.astype(int)}"
                if fmt not in WRAPPERS:
                    d_m = torch.full((n,), 7, dtype=torch.uint8, device=dev)
                    torch.cuda.synchronize(dev)   # (the calls run on the library's stream)
                    codec.is_match_device(fmt, d_src, d_off, d_len, d_m, opts)
                    torch.cuda.synchronize(dev)
                    assert np.array_equal(d_m.cpu().numpy().astype(bool), want) and int(d_m.max()) <= 1, f"{fmt_id(fmt)} {what}: device IsMatch"
            if size_fmt:
                size, st = codec.decoded_size_packed(fmt, src, off, ln, opts, size_scan=scan)
                for i, b in enumerate(blobs):
                    if b not in memo_s:
                        s1, t1 = codec.decoded_size_batch(fmt, [b], opts, size_scan=scan)
                        memo_s[b] = (int(s1[0]), int(t1[0]))
                    assert (int(size[i]), int(st[i])) == memo_s[b], f"{fmt_id(fmt)} {what}: window #{i}: size {size[i]} status {st[i]} / alone {memo_s[b]}"
                if fmt not in WRAPPERS:
                    d_size = torch.full((n,), -1, dtype=torch.int64, device=dev)
                    d_st = torch.full((n,), -9, dtype=torch.int32, device=dev)
                    torch.cuda.synchronize(dev)
                    codec.decoded_size_device(fmt, d_src, d_off, d_len, d_size, d_st, opts, size_scan=scan)
                    torch.cuda.synchronize(dev)
                    assert np.array_equal(d_size.cpu().numpy().astype(np.uint64), size) and np.array_equal(d_st.cpu().numpy(), st), \
                        f"{fmt_id(fmt)} {what}: device GetDecompressedSize"
            torch.cuda.synchronize(dev)
            assert np.array_equal(src, before) and np.array_equal(d_src.cpu().numpy(), before), f"{fmt_id(fmt)} {what}: the source changed"


# ------------------------------------------------------------------------------------------------------------ big batches
@pytest.mark.parametrize("fmt", [A.FMT_LZ10, A.FMT_LZ4_BLOCK], ids=fmt_id)
def test_pipelined_host_decode_of_repeated_windows(codec, oracle, fmt):
    """96 windows over 6 files of 768 KiB (72 MiB of capacity): the host entry point cuts the batch into pieces whose uploads
    overlap the previous pieces' windows"""
    rng = np.random.default_rng(4400 + fmt)
    raws = [synth(rng, 768 << 10, k % 5) for k in range(6)]
    comps = [oracle.encode(fmt, r, A.make_opts(quality=4))[0] for r in raws]
    image, starts = place(comps)
    pick = [int(k) for k in rng.integers(0, 6, size=96)]
    src = np.frombuffer(image + bytes(16), dtype=np.uint8).copy()
    off = np.array([starts[k] for k in pick], dtype=np.uint64)
    ln = np.array([len(comps[k]) for k in pick], dtype=np.uint64)
    caps, doff, total = layout([len(raws[k]) for k in pick])
    assert len(src) + total > (64 << 20) and len(pick) >= 64
    before = src.copy()
    dst = np.full(total + 64, SENTINEL, dtype=np.uint8)
    olen, cons, st = codec.decode_packed(fmt, src, off, ln, dst, doff, caps)
    assert np.array_equal(src, before)
    for i, k in enumerate(pick):
        assert st[i] == A.OK and olen[i] == len(raws[k]) and cons[i] == len(comps[k]), (i, st[i])
        assert dst[int(doff[i]):int(doff[i]) + len(raws[k])].tobytes() == raws[k], f"{fmt_id(fmt)}: window #{i} (file {k})"


def test_shared_windows_split_across_devices(codec, oracle):
    if codec.device_count < 2:
        pytest.skip("one device in the context")
    rng = np.random.default_rng(4500)
    raws = [synth(rng, 9000 + 1000 * k, k % 5) for k in range(3)]
    for fmt in (A.FMT_LZ00, A.FMT_LZ10, A.FMT_GCLZ):
        opts = A.make_opts(quality=8)
        comps = [oracle.encode(fmt, r, opts)[0] for r in raws]
        image, starts = place(comps)
        wins = [(s, len(image) - s) for s in starts] * 8   # the scan chain, 8 times: every device gets every window
        alone = Alone(codec, oracle, fmt, opts)
        for name, src, off, ln in variants(image, wins):
            caps, doff, total = layout([12000] * len(off))
            dst = np.full(total + 64, SENTINEL, dtype=np.uint8)
            olen, cons, st = codec.decode_packed(fmt, src, off, ln, dst, doff, caps, opts)
            compare_decode(fmt, name + " (2+ devices)", alone, src, off, ln, caps, doff, dst, olen, cons, st)
    for fmt in (A.FMT_BLZ, A.FMT_LZ00):
        memo = {}
        buf = synth(rng, 12000, 2)
        wins = [(0, 12000), (0, 6000), (16, 8000), (0, 0)] * 8
        for name, src, off, ln in variants(buf, wins):
            caps, doff, total = layout([encode_bound(codec, fmt, int(x)) for x in ln])
            dst = np.full(total + 64, SENTINEL, dtype=np.uint8)
            olen, st = codec.encode_packed(fmt, src, off, ln, dst, doff, caps, A.make_opts(quality=8))
            for i in range(len(off)):
                raw = src[int(off[i]):int(off[i]) + int(ln[i])].tobytes()
                ref, rst = memo.setdefault(raw, oracle.encode(fmt, raw, A.make_opts(quality=8)))
                assert st[i] == rst and (st[i] != A.OK or dst[int(doff[i]):int(doff[i]) + int(olen[i])].tobytes() == ref), (fmt_id(fmt), name, i)
