"""Shared helpers for the parity tests: seeded synthetic inputs and corruption operators."""
import numpy as np

from auroralib.compression_b200 import _abi as A

ALL_FORMATS = [A.FMT_YAZ0, A.FMT_YAZ1, A.FMT_YAY0, A.FMT_MIO0, A.FMT_LZ10, A.FMT_LZ11, A.FMT_LZSS, A.FMT_LZ4,
               A.FMT_LZ4_LEGACY, A.FMT_LZ4_BLOCK, A.FMT_LZO, A.FMT_SNAPPY, A.FMT_SNAPPY_BLOCK, A.FMT_PRS, A.FMT_LZHUDSON, A.FMT_LZ40, A.FMT_LZ60, A.FMT_SMSR00, A.FMT_BLZ]
MATCHABLE = [f for f in ALL_FORMATS if f not in (A.FMT_LZ4_BLOCK, A.FMT_SNAPPY_BLOCK)]   # the formats with an IsMatch rule
SIZED_FORMATS = [A.FMT_YAZ0, A.FMT_YAZ1, A.FMT_YAY0, A.FMT_MIO0, A.FMT_LZ10, A.FMT_LZ11, A.FMT_LZSS, A.FMT_LZHUDSON, A.FMT_LZ40, A.FMT_LZ60, A.FMT_SMSR00, A.FMT_BLZ]


def fmt_id(f):
    return A.FORMAT_NAMES[f]


def end_position(fmt, comp):
    """source.Position after a successful Decompress: the end of the stream, except BLZ, which reads its codes from the middle
    of the stream and leaves the position in front of the padding and the footer (BLZ.cs:56-62)."""
    return len(comp) - comp[-5] if fmt == A.FMT_BLZ else len(comp)


def synth(rng, n, kind):
    """Small asset-like buffers: 0 tiles, 1 u16 tilemap runs, 2 mixed entropy, 3 zeros/runs, 4 random."""
    if n == 0:
        return b""
    if kind == 0:
        tiles = rng.integers(0, 256, size=(16, 32), dtype=np.uint8)
        picks = rng.integers(0, 16, size=(n + 31) // 32)
        return tiles[picks].reshape(-1)[:n].tobytes()
    if kind == 1:
        out = np.zeros((n + 1) // 2, dtype=np.uint16)
        i = 0
        while i < len(out):
            run = int(rng.geometric(1 / 24))
            base = int(rng.integers(0, 1024))
            inc = int(rng.integers(0, 2))
            k = min(run, len(out) - i)
            out[i:i + k] = (base + inc * np.arange(k)) & 0x3FF | (int(rng.integers(0, 4)) << 10)
            i += k
        return out.tobytes()[:n]
    if kind == 2:
        parts = []
        total = 0
        while total < n:
            seg = int(rng.integers(16, 600))
            t = int(rng.integers(0, 3))
            if t == 0:
                p = rng.integers(0, 256, size=seg, dtype=np.uint8).tobytes()
            elif t == 1:
                p = bytes(seg)
            else:
                m = rng.integers(0, 256, size=int(rng.integers(1, 40)), dtype=np.uint8).tobytes()
                p = (m * (seg // len(m) + 1))[:seg]
            parts.append(p)
            total += seg
        return b"".join(parts)[:n]
    if kind == 3:
        out = bytearray(n)
        i = 0
        while i < n:
            run = int(rng.integers(1, 700))
            v = int(rng.integers(0, 4))
            out[i:i + run] = bytes([v]) * min(run, n - i)
            i += run
        return bytes(out[:n])
    return rng.integers(0, 256, size=n, dtype=np.uint8).tobytes()


def corrupt(rng, blob, mode):
    """0 truncate, 1 flip a byte, 2 append garbage, 3 empty, 4 cut inside the header."""
    b = bytearray(blob)
    if mode == 0 and len(b) > 1:
        return bytes(b[:int(rng.integers(1, len(b)))])
    if mode == 1 and len(b) > 0:
        i = int(rng.integers(0, len(b)))
        b[i] ^= int(rng.integers(1, 256))
        return bytes(b)
    if mode == 2:
        return bytes(b) + rng.integers(0, 256, size=int(rng.integers(1, 40)), dtype=np.uint8).tobytes()
    if mode == 3:
        return b""
    if mode == 4:
        return bytes(b[:int(rng.integers(0, min(17, len(b) + 1)))])
    return bytes(b)


def is_match_blobs(oracle, bmp, fmt):
    """IsMatch inputs for one format: oracle streams of it and of the other formats, each also corrupted, the raw data, and
    short / zero / header-only edge blobs."""
    rng = np.random.default_rng(500 + fmt)
    blobs = []
    for i in range(120):
        raw = synth(rng, int(rng.integers(5, 6000)), i % 5)
        for f in (fmt, ALL_FORMATS[i % len(ALL_FORMATS)]):
            c, st = oracle.encode(f, raw, A.make_opts(quality=int(rng.choice([0, 8]))))
            if st == 0:
                blobs.append(c)
                blobs.append(corrupt(rng, c, i % 5))
        blobs.append(raw)
    return blobs + [b"", b"\x10", b"\x10\x00\x00\x00", bmp[:300], bytes(64), bytes([0x10, 5, 0, 0, 0, 1, 2, 3, 4, 5]), bytes([0x11] + [0] * 20)]


def decoded_size_blobs(oracle, fmt):
    """GetDecompressedSize inputs for one format: oracle streams in both byte orders, cut inside the header or with a byte flipped."""
    rng = np.random.default_rng(600 + fmt)
    blobs = []
    for i in range(60):
        raw = synth(rng, int(rng.integers(1, 3000)), i % 5)
        for order in (A.ENDIAN_BIG, A.ENDIAN_LITTLE):
            c, st = oracle.encode(fmt, raw, A.make_opts(quality=0, byte_order=order))
            blobs += [c, corrupt(rng, c, 4), corrupt(rng, c, 1)]
    return blobs


def rom_like_image(oracle, rng, fmt, assets):
    """The CLI's `-scan` input: `assets` compressed at quality 8 between runs of junk -> (image, start offset of each asset)."""
    image = bytearray(rng.integers(0, 256, size=700, dtype=np.uint8).tobytes())
    starts = []
    for a in assets:
        c, st = oracle.encode(fmt, a, A.make_opts(quality=8))
        assert st == 0
        starts.append(len(image))
        image += c + rng.integers(0, 256, size=int(rng.integers(10, 400)), dtype=np.uint8).tobytes()
    return bytes(image), starts
