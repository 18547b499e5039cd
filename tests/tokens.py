"""Token programs, stream writers and seeded edge generators for the decoders.

A token program is a list of `Lit(bytes)` and `Match(distance, length)` items.  One writer per core format turns a program into a
stream of that format, choosing among the forms the format has for the same token (LZO M1 / M2 / M3 / M4, Snappy copy-1 / -2 /
-4 and literal tags 60-63, PRS short / long / long with a length byte, LZ4's optional closing literal token, MIO0 / Yay0 section
order, gaps and overlaps).  The token layouts are read from the oracle decoders (oracle/formats_*.cpp), not from the encoders,
so the streams carry the parts of each grammar that the reference encoder never writes.  `replay` restates what a program
decodes to, byte by byte, with the format's prehistory rule (zeros, or LZSS's initial fill).

`generate(fmt, rng, profile)` draws one stream from a named edge profile; `classify` counts what a program contains (distances,
periods, iteration match counts, literal spans, chains, long tokens), which the suite uses to check that every profile still
reaches its edges."""
import os
import random
import re
from collections import Counter, namedtuple

import numpy as np

from auroralib.compression_b200 import _abi as A

Lit = namedtuple("Lit", "data")
Match = namedtuple("Match", "distance length")
# one generated stream: `program` is a list of blocks (one for most formats; LZ4 legacy and Snappy framed decode each block
# with a fresh window); `expect` is the replayed output, or None when the program is meant to be rejected
Stream = namedtuple("Stream", "fmt data program expect opts lzss fill marks forms profile")

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "auroralib", "compression_b200", "csrc")


def _constants(name):
    """`#define AURORA_X n` and `constexpr int kX = <expr>;` of a kernel file, evaluated in order (expressions that name
    template parameters are skipped).  `constexpr int kA = 1, kB = kA - 1;` declares both."""
    src = re.sub(r"//[^\n]*", "", open(os.path.join(CSRC, name)).read())
    env = {}
    for m in re.finditer(r"#define (AURORA_\w+) (\d+)\b|constexpr int (k\w+ = [^;]+);", src):
        if m.group(1):
            env.setdefault(m.group(1), int(m.group(2)))
            continue
        for decl in re.split(r",\s*(?=k\w+ = )", m.group(3)):
            name, expr = decl.split(" = ", 1)
            try:
                env.setdefault(name, int(eval(expr, {"__builtins__": {}}, dict(env))))
            except Exception:
                pass
    return env


FLAG = _constants("decode_flaglz.cu")
HANDOFF_AT, ITER_MATCHES, HANDOFF_SPAN = FLAG["kHandoffAt"], FLAG["kIterMatches"], FLAG["kHandoffSpan"]
FLAG_RING, FLAG_DRAIN = FLAG["kRing"], FLAG["kFlush"]
BYTE = _constants("decode_bytelz.cu")
BYTE_KEEP, BYTE_RING, BYTE_PIECE = BYTE["kOKeep"], BYTE["kORing"], BYTE["kOPiece"]
ITER_TOKENS = 256   # tokens of one parser iteration: 32 flag groups of 8

FLAG_FORMATS = [A.FMT_LZ10, A.FMT_LZ11, A.FMT_LZ40, A.FMT_LZ60, A.FMT_YAZ0, A.FMT_YAZ1, A.FMT_LZSS, A.FMT_MIO0, A.FMT_YAY0,
                A.FMT_LZHUDSON, A.FMT_SMSR00]
BYTE_FORMATS = [A.FMT_LZ4_BLOCK, A.FMT_LZ4_LEGACY, A.FMT_LZ4, A.FMT_SNAPPY_BLOCK, A.FMT_SNAPPY, A.FMT_LZO, A.FMT_PRS]
ALL = FLAG_FORMATS + BYTE_FORMATS + [A.FMT_BLZ]
LZSS_PROPS = [(12, 4, 2), (10, 6, 2), (11, 5, 1), (8, 8, 2), ("w", 0x1000, 18, 3, 0xFEE)]

# per format: shortest and longest match, largest distance, smallest distance, whether a distance past the start of the
# output is valid (reads the prehistory) or rejected (BLZ; Snappy rejects only distances past its 64 KiB window)
Spec = namedtuple("Spec", "lo hi dmax dmin past")
SPEC = {A.FMT_LZ10: Spec(3, 18, 4096, 1, True), A.FMT_MIO0: Spec(3, 18, 4096, 1, True), A.FMT_SMSR00: Spec(3, 18, 4096, 1, True),
        A.FMT_LZ11: Spec(3, 65808, 4096, 1, True), A.FMT_LZ40: Spec(2, 65807, 4096, 1, True), A.FMT_LZ60: Spec(2, 65807, 4096, 1, True),
        A.FMT_YAZ0: Spec(3, 273, 4096, 1, True), A.FMT_YAZ1: Spec(3, 273, 4096, 1, True), A.FMT_YAY0: Spec(3, 273, 4096, 1, True),
        A.FMT_LZHUDSON: Spec(3, 273, 4096, 1, True), A.FMT_BLZ: Spec(3, 18, 4098, 3, False),
        A.FMT_LZ4_BLOCK: Spec(4, 1 << 17, 65535, 1, True), A.FMT_LZ4_LEGACY: Spec(4, 1 << 17, 65535, 1, True),
        A.FMT_LZ4: Spec(4, 1 << 17, 65535, 1, True), A.FMT_LZO: Spec(3, 1 << 16, 49151, 1, True),
        A.FMT_SNAPPY_BLOCK: Spec(1, 64, 65536, 1, True), A.FMT_SNAPPY: Spec(1, 64, 65536, 1, True),
        A.FMT_PRS: Spec(1, 256, 8192, 1, True)}


def lzss_props(p):
    return A.lz_props_window(*p[1:]) if p[0] == "w" else A.lz_props_bits(*p)


def lzss_spec(p):
    return spec_of(A.FMT_LZSS, lzss_props(p))


def spec_of(fmt, lz=None):
    if fmt != A.FMT_LZSS:
        return SPEC[fmt]
    return Spec(lz.min_length, lz.min_length + (1 << lz.length_bits) - 1, 1 << lz.windows_bits, 1, True)


# ---------------------------------------------------------------------------------------------------------------- replay
def replay(program, prehistory=0):
    """The bytes a program decodes to: literals appended, each match byte read from `distance` bytes back (copied in pieces of
    at most `distance` bytes, which is the same); bytes before the start of the output read `prehistory` (0, or LZSS's
    initial fill)."""
    out = bytearray()
    for it in program:
        if isinstance(it, Lit):
            out += it.data
            continue
        d, n = it
        k = min(n, max(d - len(out), 0))   # the bytes before the start of the output
        out += bytes([prehistory]) * k
        n -= k
        while n:
            k = min(n, d)   # a copy of at most `distance` bytes reads only bytes already written
            out += out[len(out) - d:len(out) - d + k]
            n -= k
    return bytes(out)


def merge_lits(program):
    out = []
    for it in program:
        if isinstance(it, Lit) and out and isinstance(out[-1], Lit):
            out[-1] = Lit(out[-1].data + it.data)
        elif not (isinstance(it, Lit) and not it.data):
            out.append(it)
    return out


def out_len(program):
    return sum(len(it.data) if isinstance(it, Lit) else it.length for it in program)


# ---------------------------------------------------------------------------------------------------------------- writers
class FlagOut:
    """Token bytes with flag units placed where a lazy flag reader (FlagReader.cs) fetches them: a new unit goes in front of
    the first token that needs one of its bits."""

    def __init__(self, unit=1, msb_first=True, big_endian=True, negate=False):
        self.buf, self.unit, self.msb, self.be, self.neg = bytearray(), unit, msb_first, big_endian, negate
        self.at, self.left, self.cur = 0, 0, 0

    def _store(self):
        v = self.cur
        if self.neg:
            v = -v & 0xFF
        self.buf[self.at:self.at + self.unit] = v.to_bytes(self.unit, "big" if self.be else "little")

    def bit(self, b):
        if self.left == 0:
            self.at, self.left, self.cur = len(self.buf), 8 * self.unit, 0
            self.buf += bytes(self.unit)
        self.left -= 1
        if b:
            self.cur |= 1 << (self.left if self.msb else 8 * self.unit - 1 - self.left)
        self._store()

    def run(self, one, count, data=b""):
        """`count` tokens of flag bit `one` (literals: `data` holds their bytes, placed behind their unit)"""
        i = 0
        while i < count:
            self.bit(one)
            k = min(self.left, count - i - 1)
            if one and k:
                self.cur |= ((1 << k) - 1) << (self.left - k if self.msb else 8 * self.unit - self.left)
                self._store()
            self.left -= k
            if data:
                self.buf += data[i:i + k + 1]
            i += k + 1

    def lits(self, data, one):
        self.run(one, len(data), data)


def _hdr_lz1x(ident, n):
    return bytes([ident]) + n.to_bytes(3, "little") if 0 < n <= 0xFFFFFF else bytes([ident, 0, 0, 0]) + n.to_bytes(4, "little")


def _w_flag_single(fmt, program, rng, forms, lzss=None):
    """the formats whose flags, codes and literals share one stream: LZ10, LZ11, LZ40 / LZ60, Yaz0 / Yaz1, LZHudson, LZSS"""
    lit_one = fmt in (A.FMT_YAZ0, A.FMT_YAZ1, A.FMT_LZHUDSON, A.FMT_LZSS)
    if fmt == A.FMT_LZHUDSON:
        f = FlagOut(unit=4)
    elif fmt == A.FMT_LZSS:
        f = FlagOut(msb_first=False)
    else:
        f = FlagOut(negate=fmt in (A.FMT_LZ40, A.FMT_LZ60))
    marks, pos = [], 0
    for it in program:
        if isinstance(it, Lit):
            f.lits(it.data, lit_one)
            pos += len(it.data)
            marks.append(len(f.buf))
            continue
        d, ln = it
        f.bit(not lit_one)
        if fmt == A.FMT_LZ10:
            f.buf += bytes([(ln - 3) << 4 | (d - 1) >> 8, (d - 1) & 0xFF])
        elif fmt == A.FMT_LZ11:
            if ln <= 16:
                f.buf += bytes([(ln - 1) << 4 | (d - 1) >> 8, (d - 1) & 0xFF])
                forms["lz11_2"] += 1
            elif ln <= 272:
                v = ln - 17
                f.buf += bytes([v >> 4, (v & 0xF) << 4 | (d - 1) >> 8, (d - 1) & 0xFF])
                forms["lz11_3"] += 1
            else:
                v = ln - 273
                f.buf += bytes([0x10 | v >> 12, (v >> 4) & 0xFF, (v & 0xF) << 4 | (d - 1) >> 8, (d - 1) & 0xFF])
                forms["lz11_4"] += 1
        elif fmt in (A.FMT_LZ40, A.FMT_LZ60):
            dd = d & 0xFFF   # a distance of 4096 is written as 0
            forms["lz40_d0"] += dd == 0
            if ln < 16:
                f.buf += (dd << 4 | ln).to_bytes(2, "little")
            elif ln < 272:
                f.buf += (dd << 4).to_bytes(2, "little") + bytes([ln - 16])
            else:
                f.buf += (dd << 4 | 1).to_bytes(2, "little") + (ln - 272).to_bytes(2, "little")
        elif fmt == A.FMT_LZSS:
            lz = lzss
            off = (lz.windows_start + pos - d) & (lz.max_distance - 1)
            # (a u16 token: with windows_bits + length_bits > 16 the offset's top bits are dropped, as LZSS.cs writes them)
            f.buf += (((off & 0xFF) | (off & 0xFF00) << lz.length_bits | (ln - lz.min_length) << 8) & 0xFFFF).to_bytes(2, "little")
        else:   # Yaz0 / Yaz1 / LZHudson
            if ln < 18:
                f.buf += bytes([(ln - 2) << 4 | (d - 1) >> 8, (d - 1) & 0xFF])
            else:
                f.buf += bytes([(d - 1) >> 8, (d - 1) & 0xFF, ln - 0x12])
        pos += ln
        marks.append(len(f.buf))
    return f.buf, marks


def w_lz10(program, rng, forms, ident=0x10, fmt=A.FMT_LZ10):
    body, marks = _w_flag_single(fmt, program, rng, forms)
    h = _hdr_lz1x(ident, out_len(program))
    return h + body, [len(h) + m for m in marks]


def w_yaz0(program, rng, forms, magic, order):
    n = out_len(program)
    bo = "little" if order == A.ENDIAN_LITTLE else "big"
    h = magic + n.to_bytes(4, bo) + int(rng.choice([0, 0x20, 0x80])).to_bytes(4, bo) + bytes(4)
    body, marks = _w_flag_single(A.FMT_YAZ0, program, rng, forms)
    return h + body, [len(h) + m for m in marks]


def w_lzhudson(program, rng, forms):
    body, marks = _w_flag_single(A.FMT_LZHUDSON, program, rng, forms)
    return out_len(program).to_bytes(4, "big") + body, [4 + m for m in marks]


def w_lzss(program, rng, forms, lz):
    n = out_len(program)
    body, marks = _w_flag_single(A.FMT_LZSS, program, rng, forms, lzss=lz)
    return b"LZSS" + n.to_bytes(4, "big") + len(body).to_bytes(4, "big") + bytes(4) + body, [16 + m for m in marks]


def w_sections(fmt, program, rng, forms, order):
    """MIO0 / Yay0: flags at 0x10, then the code and literal sections in either order, with gaps, or overlapping where the
    bytes allow it (the overlap is made by choosing literal values).  Returns the (possibly re-valued) program too."""
    flags, codes, lits, owner = FlagOut(), bytearray(), bytearray(), []
    prog = [Lit(bytearray(it.data)) if isinstance(it, Lit) else it for it in program]
    for k, it in enumerate(prog):
        if isinstance(it, Lit):
            flags.run(1, len(it.data))
            lits += it.data
            owner += [(k, j) for j in range(len(it.data))]
            continue
        d, ln = it
        flags.bit(0)
        if fmt == A.FMT_MIO0 or ln < 18:
            codes += ((ln - (3 if fmt == A.FMT_MIO0 else 2)) << 12 | (d - 1)).to_bytes(2, "big")
        else:
            codes += (d - 1).to_bytes(2, "big")
            lits.append(ln - 0x12)
            owner.append(None)
    layout = rng.choice(["codes_lits", "lits_codes", "gaps", "overlap"]) if rng.random() < 0.7 else "codes_lits"
    first, second = (lits, codes) if layout == "lits_codes" or (layout in ("gaps", "overlap") and rng.random() < 0.5) else (codes, lits)
    gap0, gap1 = (int(rng.integers(1, 40)), int(rng.integers(1, 40))) if layout == "gaps" else (0, 0)
    ov = 0
    if layout == "overlap" and len(first) and len(second):
        # second[:ov] must equal first[-ov:]; the literal section's free bytes are set to make it so
        want = int(rng.integers(1, 9))
        for k in range(min(want, len(first), len(second)), 0, -1):
            idx_l = range(len(lits) - k, len(lits)) if first is lits else range(k)
            if all(owner[i] is not None for i in idx_l):
                for t in range(k):
                    if first is lits:
                        i = len(lits) - k + t
                        lits[i] = codes[t]
                    else:
                        i = t
                        lits[i] = codes[len(codes) - k + t]
                    ki, j = owner[i]
                    prog[ki].data[j] = lits[i]
                ov = k
                break
    forms[f"layout_{layout if layout != 'overlap' or ov else 'codes_lits'}"] += 1
    forms["lits_first"] += first is lits
    p_first = 0x10 + len(flags.buf) + gap0
    p_second = p_first + len(first) - ov + gap1
    p_codes, p_lits = (p_first, p_second) if first is codes else (p_second, p_first)
    bo = "little" if order == A.ENDIAN_LITTLE else "big"
    n = out_len(program)
    junk = lambda k: rng.integers(0, 256, size=k, dtype=np.uint8).tobytes()
    data = (fmt == A.FMT_MIO0 and b"MIO0" or b"Yay0") + n.to_bytes(4, bo) + p_codes.to_bytes(4, bo) + p_lits.to_bytes(4, bo)
    data += flags.buf + junk(gap0) + first + junk(gap1) + second[ov:] + junk(int(rng.integers(0, 3)) * (layout == "gaps"))
    prog = [Lit(bytes(it.data)) if isinstance(it, Lit) else it for it in prog]
    return bytes(data), [], prog


def w_smsr00(program, rng, forms):
    f, lits = FlagOut(unit=2), bytearray()
    for it in program:
        if isinstance(it, Lit):
            f.run(1, len(it.data))
            lits += it.data
        else:
            f.bit(0)
            f.buf += ((it.length - 3) << 12 | (it.distance - 1)).to_bytes(2, "big")
    pad = int(rng.choice([0, 0, 1, 2]))   # trailing bytes of the code section: an odd one is not addressable
    forms[f"smsr_pad{pad}"] += 1
    codes = f.buf + bytes(pad)
    return b"SMSR00" + bytes(2) + out_len(program).to_bytes(4, "big") + (0x10 + len(codes)).to_bytes(4, "big") + codes + lits, []


def w_blz(program, rng, forms):
    """BLZ is read from its end: flag bytes (MSB first, 1 = match), literals and (length - 3) << 12 | (distance - 3) codes,
    high byte first, all in reverse; the program describes the output from its last byte backwards."""
    f = FlagOut()
    for it in program:
        if isinstance(it, Lit):
            f.lits(it.data, 0)
        else:
            f.bit(1)
            info = (it.length - 3) << 12 | (it.distance - 3)
            f.buf += bytes([info >> 8, info & 0xFF])
    codes = bytes(f.buf[::-1])
    pad = int(rng.choice([(16 - (len(codes) + 8) % 16) % 16, 0, 5]))
    comp = len(codes) + pad + 8
    n = out_len(program)
    return codes + b"\xff" * pad + comp.to_bytes(3, "little") + bytes([pad + 8]) + ((n - comp) & 0xFFFFFFFF).to_bytes(4, "little"), []


def _lz4_ext(v):
    out = bytearray()
    while True:
        b = min(v, 255)
        out.append(b)
        v -= b
        if b != 255:
            return out


def w_lz4_block(program, rng, forms):
    out, marks, pend = bytearray(), [], b""
    for k, it in enumerate(program):
        if isinstance(it, Lit):
            pend += it.data
            continue
        lit, m = len(pend), it.length - 4
        out.append(min(lit, 15) << 4 | min(m, 15))
        if lit >= 15:
            out += _lz4_ext(lit - 15)
        out += pend + it.distance.to_bytes(2, "little")
        if m >= 15:
            out += _lz4_ext(m - 15)
        pend = b""
        marks.append(len(out))
    if pend or rng.random() < 0.5:   # a block may end right after a match (LZ4.cs:189 breaks at the end of the input)
        forms["lz4_literal_tail"] += 1
        out.append(min(len(pend), 15) << 4)
        if len(pend) >= 15:
            out += _lz4_ext(len(pend) - 15)
        out += pend
    else:
        forms["lz4_match_tail"] += 1
    return out, marks


def w_lz4_legacy(blocks, rng, forms):
    out = bytearray((0x184C2102).to_bytes(4, "little"))
    for k, b in enumerate(blocks):
        body, _ = w_lz4_block(b, rng, forms)
        assert not (k and len(body) & 0xFF == 0xFF), "LZ4.cs:103 reads a block size that starts with 0xFF as the end mark"
        out += len(body).to_bytes(4, "little") + body
    if rng.random() < 0.5:
        out.append(0xFF)
    return bytes(out), []


def w_lz4_frame(blocks, rng, forms, oracle):
    """one v1 frame, blocks linked (one window across the frame); some blocks stored; optional content size"""
    n = sum(out_len(b) for b in blocks)
    flg = 0x40 | (0x08 if rng.random() < 0.3 else 0)
    bd = 0x70
    desc = bytes([flg, bd]) + (n.to_bytes(8, "little") if flg & 8 else b"")
    out = bytearray((0x184D2204).to_bytes(4, "little")) + desc + bytes([(oracle.xxh32(desc) >> 8) & 0xFF])
    done = []
    for b in blocks:
        if rng.random() < 0.15:
            raw = replay(done + b)[out_len(done):]
            out += (len(raw) | 0x80000000).to_bytes(4, "little") + raw
            forms["lz4_stored_block"] += 1
        else:
            body, _ = w_lz4_block(b, rng, forms)
            out += len(body).to_bytes(4, "little") + body
        done += b
    out += bytes(4)
    return bytes(out), []


def _varint(v):
    out = bytearray()
    while v >= 0x80:
        out.append(v & 0x7F | 0x80)
        v >>= 7
    out.append(v)
    return out


def w_snappy_block(program, rng, forms):
    out, marks = bytearray(_varint(out_len(program))), []
    for it in program:
        if isinstance(it, Lit):
            L = len(it.data) - 1
            need = 0 if L < 60 else 1 if L <= 0xFF else 2 if L <= 0xFFFF else 3 if L <= 0xFFFFFF else 4
            if need == 0 and rng.random() < 0.7:
                out.append(L << 2)
            else:   # tags 60-63: 1-4 length bytes, also more than the length needs
                tag = 59 + int(rng.integers(max(need, 1), 5))
                out.append(tag << 2)
                out += L.to_bytes(tag - 59, "little")
                forms[f"snappy_tag{tag}"] += 1
            out += it.data
        else:
            d, ln = it
            c = ["c4"]
            if ln <= 64 and d <= 0xFFFF:
                c.append("c2")
            if 4 <= ln <= 11 and d < 2048:
                c += ["c1", "c1"]
            form = c[int(rng.integers(0, len(c)))]
            forms["snappy_" + form] += 1
            if form == "c1":
                out += bytes([1 | (ln - 4) << 2 | (d >> 8) << 5, d & 0xFF])
            elif form == "c2":
                out += bytes([2 | (ln - 1) << 2]) + d.to_bytes(2, "little")
            else:
                out += bytes([3 | (ln - 1) << 2]) + d.to_bytes(4, "little")
        marks.append(len(out))
    return out, marks


def w_snappy_framed(blocks, rng, forms):
    out = bytearray(b"\xff\x06\x00\x00sNaPpY")
    for b in blocks:
        if rng.random() < 0.15:
            out += bytes([0xFE]) + (3).to_bytes(3, "little") + b"pad"   # a skippable chunk
            forms["snappy_skip_chunk"] += 1
        if rng.random() < 0.15:
            raw = replay(b)
            out += bytes([1]) + (len(raw) + 4).to_bytes(3, "little") + bytes(4) + raw
            forms["snappy_stored_chunk"] += 1
        else:
            body, _ = w_snappy_block(b, rng, forms)
            out += bytes([0]) + (len(body) + 4).to_bytes(3, "little") + bytes(4) + body
    return bytes(out), []


def _lzo_ext(v):
    out = bytearray()
    while v > 255:
        out.append(0)
        v -= 255
    out.append(v)
    return out


def w_lzo(program, rng, forms):
    """The decoder's state (LZO.cs:49-139): after a literal run a 0x0X flag is a 3-byte match at distance 2049-3072; after a
    match with 1-3 trailing literals it is a 2-byte M1 match (distance 1-1024); otherwise it starts a literal run."""
    prog = merge_lits(program)
    out, marks, state, k = bytearray(), [], 0, 0
    if prog and isinstance(prog[0], Lit) and (len(prog[0].data) < 4 or (len(prog[0].data) <= 238 and rng.random() < 0.5)):
        out.append(17 + len(prog[0].data))
        out += prog[0].data
        forms["lzo_first_byte_run"] += 1
        k = 1
        marks.append(len(out))
    while k < len(prog):
        it = prog[k]
        if isinstance(it, Lit):
            L = len(it.data)
            assert L >= 4 and state == 0, "a literal run needs 4 bytes and a state of 0"
            out += bytes([L - 3]) if L <= 18 else bytes([0]) + _lzo_ext(L - 18)
            out += it.data
            state = 4
            k += 1
            marks.append(len(out))
            continue
        d, ln = it
        t = 0
        if k + 1 < len(prog) and isinstance(prog[k + 1], Lit) and len(prog[k + 1].data) <= 3:
            t = len(prog[k + 1].data)
        c = []
        if ln == 2 and 1 <= state <= 3 and d <= 1024:
            c.append("m1")
        if ln == 3 and state == 4 and 2049 <= d <= 3072:
            c.append("m1_far")
        if 3 <= ln <= 8 and d <= 2048:
            c.append("m2")
        if ln >= 3 and d <= 16384:
            c.append("m3")
        if ln >= 3 and 16385 <= d <= 49151:
            c.append("m4")
        assert c, f"LZO cannot write Match({d}, {ln}) in state {state}"
        form = c[int(rng.integers(0, len(c)))]
        forms["lzo_" + form] += 1
        if form == "m1":
            out += bytes([((d - 1) & 3) << 2 | t, (d - 1) >> 2])
        elif form == "m1_far":
            x = d - 2049
            out += bytes([(x & 3) << 2 | t, x >> 2])
        elif form == "m2":
            hi = 0x40 | (ln - 3) << 5 if ln <= 4 else 0x80 | (ln - 5) << 5
            out += bytes([hi | ((d - 1) & 7) << 2 | t, (d - 1) >> 3])
        elif form == "m3":
            out += bytes([0x20 | (ln - 2)]) if ln <= 33 else bytes([0x20]) + _lzo_ext(ln - 33)
            out += bytes([((d - 1) & 0x3F) << 2 | t, (d - 1) >> 6])
        else:
            x = d - 16384
            h, x = x >> 14, x & 0x3FFF
            out += bytes([0x10 | h << 3 | (ln - 2)]) if ln <= 9 else bytes([0x10 | h << 3]) + _lzo_ext(ln - 9)
            out += bytes([(x & 0x3F) << 2 | t, x >> 6])
        k += 1
        if t:
            out += prog[k].data
            k += 1
        state = t
        marks.append(len(out))
    out += b"\x11\x00\x00"
    return bytes(out), marks


def w_prs(program, rng, forms, order):
    be = order == A.ENDIAN_BIG
    f = FlagOut(msb_first=be)
    u16 = lambda v: v.to_bytes(2, "big" if be else "little")
    marks = []
    for it in program:
        if isinstance(it, Lit):
            f.lits(it.data, 1)
        else:
            d, ln = it
            c = []
            if 2 <= ln <= 5 and d <= 256:
                c.append("short")
            if 3 <= ln <= 9:
                c.append("long")
            if d < 8192:
                c.append("long_byte")
            form = c[int(rng.integers(0, len(c)))]
            forms["prs_" + form] += 1
            f.bit(0)
            if form == "short":
                f.bit(0)
                f.bit((ln - 2) >> 1)
                f.bit((ln - 2) & 1)
                f.buf.append((0x100 - d) & 0xFF)
            else:
                f.bit(1)
                if form == "long":
                    f.buf += u16((0x2000 - d) << 3 | (ln - 2))
                else:
                    f.buf += u16((0x2000 - d) << 3) + bytes([ln - 1])
        marks.append(len(f.buf))
    f.bit(0)
    f.bit(1)
    f.buf += bytes(2)
    return bytes(f.buf), marks


# ---------------------------------------------------------------------------------------------------------------- generators
class Builder:
    def __init__(self, rng, spec, fmt):
        self.rng, self.spec, self.fmt, self.items, self.n, self.tokens = rng, spec, fmt, [], 0, 0
        self.bytes = random.Random(int(rng.integers(1 << 62))).randbytes   # literal values (numpy per call is slow here)

    def lit(self, k):
        if k > 0:
            self.items.append(Lit(self.bytes(k)))
            self.n += k
            self.tokens += k

    def match(self, d, ln):
        self.items.append(Match(int(d), int(ln)))
        self.n += ln
        self.tokens += 1

    def rlen(self, cap=300):
        s = self.spec
        hi = max(s.lo, min(s.hi, cap))
        return int(self.rng.integers(s.lo, hi + 1)) if self.rng.random() < 0.8 else int(self.rng.integers(s.lo, min(s.lo + 3, hi) + 1))

    def rdist(self):
        s = self.spec
        top = max(s.dmin, min(self.n, s.dmax))
        r = self.rng.random()
        if r < 0.3:
            return int(self.rng.integers(s.dmin, min(top, s.dmin + 16) + 1))
        return int(self.rng.integers(s.dmin, top + 1))

    def any_match(self, cap=300):
        self.match(self.rdist(), self.rlen(cap))


def _flag_queue(b, rng):
    """iterations of exactly k matches in 256 tokens at the hand-off and queue limits, literal spans at the byte hand-off, chains
    of same-distance matches (and the same broken by one literal), pairs whose second source overlaps the first destination"""
    s = b.spec
    b.lit(int(rng.integers(300, 700)))
    b.lit((-b.tokens) % ITER_TOKENS)
    counts = [HANDOFF_AT - 1, HANDOFF_AT, HANDOFF_AT + 1, ITER_MATCHES, ITER_MATCHES + 1]
    for k in rng.permutation(counts + [int(rng.integers(0, 160))]):
        slots = set(int(x) for x in rng.choice(ITER_TOKENS, size=int(k), replace=False))
        for t in range(ITER_TOKENS):
            if t in slots:
                b.match(b.rdist(), int(rng.integers(s.lo, max(s.lo, min(s.hi, 18)) + 1)))
            else:
                b.lit(1)
    for delta in rng.permutation([-1, 0, 1]):
        b.any_match(40)
        b.lit(HANDOFF_SPAN + int(delta))
    for _ in range(int(rng.integers(2, 5))):
        d = int(rng.integers(1, 40))
        hi = min(s.hi, 18)
        for _ in range(int(rng.integers(3, 12))):
            b.match(d, int(rng.integers(s.lo, max(s.lo, hi - 1) + 1)))
        b.lit(1)
        for _ in range(int(rng.integers(2, 6))):
            b.match(d, int(rng.integers(s.lo, max(s.lo, hi - 1) + 1)))
            b.lit(1)
        l1 = int(rng.integers(s.lo, max(s.lo, min(s.hi, 40)) + 1))
        b.match(b.rdist(), l1)
        b.match(int(rng.integers(1, min(l1, s.dmax) + 1)), int(rng.integers(s.lo, max(s.lo, min(s.hi, 40)) + 1)))


def _lzo_forms(b, rng):
    """LZO's M1 forms in both states and the first-byte literal run"""
    b.lit(int(rng.integers(4, 200)))
    for _ in range(int(rng.integers(20, 80))):
        r = rng.random()
        b.any_match(60)
        if r < 0.5:
            for _ in range(int(rng.integers(1, 5))):
                b.lit(int(rng.integers(1, 4)))
                b.match(int(rng.integers(1, min(b.n, 1024) + 1)), 2)
        b.lit(int(rng.integers(1, 4)) if r < 0.7 else 0)
        if rng.random() < 0.4:
            b.lit(int(rng.integers(4, 30)))
            if b.n > 3072:
                b.match(int(rng.integers(2049, 3073)), 3)
        elif rng.random() < 0.3:
            b.lit(int(rng.integers(4, 30)))


def generate(fmt, rng, profile, size=None, oracle=None, lzss_props=None):
    """One stream of `fmt` drawn from `profile` (mixed, short_periods, window, ring, queue, long, forms).  LZSS draws its
    properties from LZSS_PROPS unless `lzss_props` names one set in the same notation."""
    lzp = None
    spec = SPEC.get(fmt)
    if fmt == A.FMT_LZSS:
        lzp = lzss_props if lzss_props is not None else LZSS_PROPS[int(rng.integers(0, len(LZSS_PROPS)))]
        spec = lzss_spec(lzp)
    b = Builder(rng, spec, fmt)
    size = size or int(rng.choice([300, 2000, 6000, 12000, 30000]))
    flag = fmt in FLAG_FORMATS
    snappy = fmt in (A.FMT_SNAPPY_BLOCK, A.FMT_SNAPPY)
    invalid = False
    start = lambda lo, hi: b.lit(int(rng.integers(max(lo, spec.dmin), max(hi, spec.dmin + 1))))   # BLZ: nothing to copy from
    if fmt == A.FMT_PRS:
        # PRS.cs:161-218 guesses the byte order from the first flag byte (odd and > 12: little; MSB set: big) and the first four
        # matches (none may reach past the start).  Seven literals and a match make the first flag byte 0x7F / 0xFE, which the
        # guess reads right in both orders.
        b.lit(7)
        for _ in range(4):
            b.match(int(rng.integers(1, b.n + 1)), int(rng.integers(3, 10)))
    if profile == "mixed":
        start(1, 64)
        while b.n < size:
            if rng.random() < 0.45:
                b.lit(int(rng.geometric(0.08)))
            else:
                b.any_match()
    elif profile == "short_periods":
        start(8, 16)
        while b.n < size:
            d = int(rng.integers(spec.dmin, spec.dmin + 4))
            lo, hi = max(spec.lo, d + 1), min(spec.hi, 600)
            if lo <= hi:
                b.match(d, int(rng.integers(lo, hi + 1)))
            if rng.random() < 0.5:
                b.lit(int(rng.integers(1, 6)))
    elif profile == "window":
        if fmt != A.FMT_BLZ and rng.random() < 0.6:   # distances past the start of the output read the prehistory
            b.lit(int(rng.integers(1, 40)))
            for _ in range(int(rng.integers(1, 4))):
                b.match(int(rng.integers(min(b.n + 1, spec.dmax), spec.dmax + 1)), b.rlen(40))
                b.lit(int(rng.integers(1, 10)))
        elif (fmt == A.FMT_BLZ or snappy) and rng.random() < 0.25:   # ... or are rejected
            b.lit(int(rng.integers(spec.dmin, 50)))
            b.match(b.n + int(rng.integers(1, 30)) if fmt == A.FMT_BLZ else spec.dmax + int(rng.integers(1, 3)), b.rlen(20))
            invalid = True
        b.lit(spec.dmax + int(rng.integers(0, 200)))
        for _ in range(int(rng.integers(5, 40))):
            b.match(max(spec.dmax - int(rng.choice([0, 0, 1, 2])), spec.dmin), b.rlen(60))
            b.lit(int(rng.integers(0, 6)))
    elif profile == "ring":
        start(20, 100)
        if flag or fmt == A.FMT_BLZ:   # matches across the 8 KiB ring wrap, totals at a drain step and one byte either side
            total = FLAG_DRAIN * int(rng.integers(1, 60)) + int(rng.choice([-1, 0, 1]))
            while b.n < total - 300:
                if rng.random() < 0.5:
                    b.match(b.rdist(), b.rlen(min(total - 300 - b.n, 2500)))
                else:
                    b.lit(int(rng.integers(1, 30)))
            b.lit(total - b.n)
        else:   # distances at the shared ring's keep and size limits, sources across a drain step
            while b.n < size:
                d = int(rng.choice([BYTE_KEEP - 1, BYTE_KEEP, BYTE_KEEP + 1, BYTE_RING - 1, BYTE_RING, BYTE_RING + 1]))
                if b.n < d:
                    b.lit(d - b.n + int(rng.integers(0, 50)))
                ln = b.rlen(80)
                if rng.random() < 0.5:
                    b.lit((-(b.n - d) - int(rng.integers(1, min(ln, d) + 1))) % BYTE_PIECE)
                b.match(d, ln)
                b.lit(int(rng.integers(0, 5)))
    elif profile == "queue":
        _flag_queue(b, rng)
    elif profile == "long":
        start(1, 5000)
        for _ in range(int(rng.integers(1, 5))):
            if spec.hi >= 65807:   # LZ11 / LZ40 / LZ60: around the 2 KiB segments of the long-message path, and the top
                k = int(rng.integers(8, 33))
                ln = int(rng.choice([2048 * k - 1, 2048 * k, 2048 * k + 1, spec.hi, spec.hi - 1, 16385]))
                ln = min(max(ln, 16385), spec.hi)
            elif fmt in (A.FMT_LZ4_BLOCK, A.FMT_LZ4_LEGACY, A.FMT_LZ4):   # 15 + 255 k - 1, + 0, + 1
                ln = 4 + 15 + 255 * int(rng.integers(0, 12)) + int(rng.choice([-1, 0, 1]))
                b.lit(15 + 255 * int(rng.integers(0, 12)) + int(rng.choice([-1, 0, 1])))
            elif fmt == A.FMT_LZO:
                ln = int(rng.choice([33, 34, 35, 9, 10, 300, 4000]))
            else:
                ln = spec.hi - int(rng.choice([0, 0, 1]))
            ds = [d for d in (1, 2, 3, 17, 4096) if spec.dmin <= d <= min(spec.dmax, b.n if fmt == A.FMT_BLZ else spec.dmax)]
            b.match(int(rng.choice(ds + [b.rdist()])), ln)
            b.lit(int(rng.integers(0, 300)))
            if snappy:   # literal lengths at the tag 60 / 61 / 62 limits
                b.lit(int(rng.choice([61, 256, 257, 65536, 65537])))
    elif profile == "forms":   # the forms the reference encoder never writes
        if fmt == A.FMT_LZO:
            _lzo_forms(b, rng)
        else:
            start(1, 600)
            while b.n < size:
                if snappy and b.n > 32768 and rng.random() < 0.3:
                    b.match(int(rng.integers(32769, min(b.n, 65536) + 1)), int(rng.integers(1, 65)))
                elif fmt == A.FMT_PRS and rng.random() < 0.4:
                    b.match(b.rdist(), int(rng.integers(1, 10)))
                elif rng.random() < 0.5:
                    b.any_match(20)
                else:
                    b.lit(int(rng.integers(1, 12)))
    else:
        raise ValueError(profile)
    prog = merge_lits(b.items)
    if fmt == A.FMT_LZO:
        prog = _lzo_fix(prog)
    elif fmt == A.FMT_PRS:   # a distance of 8192 has only the long form without a length byte (3-9 bytes)
        prog = [Match(it.distance, min(max(it.length, 3), 9)) if isinstance(it, Match) and it.distance == 8192 else it for it in prog]
    elif fmt == A.FMT_LZSS:   # a distance of the whole window copies the ring onto itself: at most one window long
        prog = [Match(it.distance, min(it.length, spec.dmax)) if isinstance(it, Match) and it.distance == spec.dmax else it for it in prog]
    return write(fmt, prog, rng, profile, invalid=invalid, lzp=lzp, oracle=oracle)


def _lzo_fix(prog):
    """LZO cannot place 1-3 literals in front of a literal run, nor a 2-byte match except right after trailing literals:
    lengthen such literals to 4 and such matches to 3"""
    out, state = [], 0
    for k, it in enumerate(prog):
        if isinstance(it, Lit):
            if len(it.data) < 4 and k > 0 and not isinstance(prog[k - 1], Match):
                it = Lit(it.data + bytes(4 - len(it.data)))
            state = len(it.data) if len(it.data) <= 3 and k > 0 else 4
        else:
            if it.length == 2 and not (1 <= state <= 3 and it.distance <= 1024):
                it = Match(it.distance, 3)
            state = 0
        out.append(it)
    return merge_lits(out)


def _split(prog, rng, parts):
    if parts <= 1 or len(prog) < 4:
        return [prog]
    cuts = sorted(set(int(x) for x in rng.integers(1, len(prog), size=parts - 1)))
    return [prog[a:b] for a, b in zip([0] + cuts, cuts + [len(prog)])]


def write(fmt, prog, rng, profile="", invalid=False, lzp=None, oracle=None):
    forms = Counter()
    opts_kw, lz, fill, marks = {}, None, 0, []
    blocks = [prog]
    if fmt in (A.FMT_LZ10, A.FMT_LZ11, A.FMT_LZ40, A.FMT_LZ60):
        data, marks = w_lz10(prog, rng, forms, {A.FMT_LZ10: 0x10, A.FMT_LZ11: 0x11, A.FMT_LZ40: 0x40, A.FMT_LZ60: 0x60}[fmt], fmt)
    elif fmt in (A.FMT_YAZ0, A.FMT_YAZ1):
        order = int(rng.choice([A.ENDIAN_BIG, A.ENDIAN_LITTLE]))
        explicit = order == A.ENDIAN_LITTLE and rng.random() < 0.7   # a little-endian header under the default order: the retry
        if explicit:
            opts_kw["byte_order"] = order
        forms[f"yaz_order{order}{'x' if explicit else ''}"] += 1
        data, marks = w_yaz0(prog, rng, forms, b"Yaz0" if fmt == A.FMT_YAZ0 else b"Yaz1", order)
    elif fmt == A.FMT_LZHUDSON:
        data, marks = w_lzhudson(prog, rng, forms)
    elif fmt == A.FMT_LZSS:
        lz = lzss_props(lzp)
        fill = int(rng.choice([0, 0, 0x20, 0xFF]))
        opts_kw.update(lzss=lz, lzss_initial_fill=fill)
        forms[f"lzss_{lzp}_fill{fill}"] += 1
        data, marks = w_lzss(prog, rng, forms, lz)
    elif fmt in (A.FMT_MIO0, A.FMT_YAY0):
        order = int(rng.choice([A.ENDIAN_BIG, A.ENDIAN_LITTLE]))
        if order == A.ENDIAN_LITTLE or rng.random() < 0.3:
            opts_kw["byte_order"] = order
        data, marks, prog = w_sections(fmt, prog, rng, forms, order)
        blocks = [prog]
    elif fmt == A.FMT_SMSR00:
        data, marks = w_smsr00(prog, rng, forms)
    elif fmt == A.FMT_BLZ:
        data, marks = w_blz(prog, rng, forms)
    elif fmt == A.FMT_LZ4_BLOCK:
        data, marks = w_lz4_block(prog, rng, forms)
    elif fmt == A.FMT_LZ4_LEGACY:
        for attempt in range(20):   # (a cut whose next block size starts with 0xFF is drawn again)
            blocks = _split(prog, rng, int(rng.integers(1, 4)) if attempt < 19 else 1)
            try:
                data, marks = w_lz4_legacy(blocks, rng, forms)
                break
            except AssertionError:
                continue
    elif fmt == A.FMT_LZ4:
        data, marks = w_lz4_frame(_split(prog, rng, int(rng.integers(1, 5))), rng, forms, oracle)   # one window: `blocks` stays [prog]
    elif fmt == A.FMT_SNAPPY_BLOCK:
        data, marks = w_snappy_block(prog, rng, forms)
    elif fmt == A.FMT_SNAPPY:
        blocks = _split(prog, rng, int(rng.integers(1, 4)))
        data, marks = w_snappy_framed(blocks, rng, forms)
    elif fmt == A.FMT_LZO:
        data, marks = w_lzo(prog, rng, forms)
    elif fmt == A.FMT_PRS:
        order = int(rng.choice([A.ENDIAN_BIG, A.ENDIAN_LITTLE]))
        forms[f"prs_order{order}"] += 1
        data, marks = w_prs(prog, rng, forms, order)
    else:
        raise ValueError(fmt)
    if invalid:
        expect = None
    else:
        expect = b"".join(replay(blk, fill) for blk in blocks)
        if fmt == A.FMT_BLZ:
            expect = expect[::-1]
    return Stream(fmt, bytes(data), blocks, expect, A.make_opts(**opts_kw), lz, fill, marks, forms, profile)


PROFILES = ["mixed", "short_periods", "window", "ring", "queue", "long", "forms"]


def profiles_of(fmt):
    return [p for p in PROFILES if p != "queue" or fmt in FLAG_FORMATS]


# ---------------------------------------------------------------------------------------------------------------- coverage
def classify(fmt, program, spec):
    """Counts of the edges a program holds, by name."""
    c = Counter()
    pos, tok, iter_matches, prev = 0, 0, 0, None
    items = merge_lits(program)
    for k, it in enumerate(items):
        if isinstance(it, Lit):
            L = len(it.data)
            if isinstance(prev, Match) and k + 1 < len(items):
                c[f"span{L - HANDOFF_SPAN:+d}"] += abs(L - HANDOFF_SPAN) <= 1
            if fmt in (A.FMT_LZ4_BLOCK, A.FMT_LZ4_LEGACY, A.FMT_LZ4) and L >= 15 and (L - 15) % 255 in (0, 1, 254):
                c["lz4_lit_ext_edge"] += 1
            # the iteration match counts: whole 256-token blocks from the start of the stream
            while L:
                step = min(L, ITER_TOKENS - tok % ITER_TOKENS)
                tok += step
                L -= step
                if tok % ITER_TOKENS == 0:
                    c[f"iter{iter_matches}"] += 1
                    iter_matches = 0
            pos += len(it.data)
            prev = it
            continue
        d, ln = it
        if d <= 4 and ln > d:
            c[f"period{d}"] += 1
        if d == spec.dmax:
            c["dmax"] += 1
        if d > pos:
            c["past_start"] += 1
        if pos // FLAG_RING != (pos + ln - 1) // FLAG_RING:
            c["ring_wrap"] += 1
        if d in (BYTE_KEEP - 1, BYTE_KEEP, BYTE_KEEP + 1, BYTE_RING - 1, BYTE_RING, BYTE_RING + 1):
            c["byte_ring_dist"] += 1
        if (pos - d) // BYTE_PIECE != (pos - d + min(ln, d) - 1) // BYTE_PIECE and d > BYTE_PIECE:
            c["source_straddles_drain"] += 1
        if ln >= 16385:
            c["len_over_16k"] += 1
            c["len_2048k"] += (ln % 2048) in (0, 1, 2047)
        if ln == spec.hi:
            c["len_max"] += 1
        if fmt in (A.FMT_LZ4_BLOCK, A.FMT_LZ4_LEGACY, A.FMT_LZ4) and ln - 4 >= 15 and (ln - 19) % 255 in (0, 1, 254):
            c["lz4_match_ext_edge"] += 1
        if isinstance(prev, Match):
            if prev.distance == d and ln < spec.hi and prev.length < spec.hi:
                c["chain"] += 1
            if d <= prev.length:
                c["overlap_pair"] += 1
        if k >= 2 and isinstance(items[k - 2], Match) and items[k - 2].distance == d and isinstance(prev, Lit) and len(prev.data) == 1:
            c["chain_broken"] += 1
        iter_matches += 1
        tok += 1
        if tok % ITER_TOKENS == 0:
            c[f"iter{iter_matches}"] += 1
            iter_matches = 0
        pos += ln
        prev = it
    if pos >= FLAG_DRAIN and pos % FLAG_DRAIN in (0, 1, FLAG_DRAIN - 1):
        c["total_at_drain_step"] += 1
    return c
