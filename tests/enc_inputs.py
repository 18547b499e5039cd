"""Raw inputs built against the encoders' match finders: the lane-per-position search of csrc/encode_lz_par.cu (its bucket
heads, tagged node ring, in-step candidates, data ring and lazy step hand-over) and the sequential replay of csrc/finder.cuh
with the byte-LZ token writers of csrc/encode_bytelz.cu.

An input is a program of fresh bytes, copies and 4-byte groups whose hash is chosen: 2654435761 is odd, so it is invertible
modulo 2^32 and a group with any wanted hash value is `(hash << (32 - hash_bits) | low) * inverse`.  Fresh bytes never repeat a
min_length-gram within the window, and never fall into a bucket that a designed group uses; `build` rejects a result in which
either happens anyway (across the seams of copies and groups), so the only matches an input holds are the planted ones.

Every profile returns `(name, a, b)` pairs of equal length that differ only across one edge (max_chain - 1 against max_chain
decoys, distance max_dist against max_dist + 1, ...): the reference encoder's outputs of the two differ in length, which the
suite checks, so an edge that stopped deciding anything shows up as a broken profile."""
import random

from auroralib.compression_b200 import _abi as A
from tests.test_simt_kernels import finder_params
from tests.tokens import _constants

PAR = _constants("encode_lz_par.cu")
BUCKET_BITS, WIN, LOOK, CHUNK, DATA = PAR["AURORA_ENC_BUCKET_BITS"], PAR["kWin"], PAR["kLook"], PAR["kChunk"], PAR["AURORA_ENC_DATA"]
BUCKET_MASK = (1 << BUCKET_BITS) - 1
PARK = 0x4000   # the heads' parking pass runs at every multiple of this position

PRIME = 2654435761
INVERSE = pow(PRIME, -1, 1 << 32)
M32 = 0xFFFFFFFF


class Params:
    """The finder parameters of one format / quality / option set (finder_params of test_simt_kernels)."""

    def __init__(self, fmt, quality, vram_mode=-1, lzss=None):
        f, _ = finder_params(fmt, quality, 0, vram_mode, lzss)
        self.fmt, self.quality = fmt, quality
        self.max_chain, self.lazy, self.hash_bits, _, self.min_len, self.max_len, self.min_dist, self.max_dist, _, self.min_table = f


def full_hash(v4, bits):
    return ((v4 * PRIME) & M32) >> (32 - bits)


def group_with_hash(h, bits, rnd):
    """Four bytes whose LzChainMatchFinder hash (ComputeHash) is h."""
    low = rnd.getrandbits(32 - bits)
    return (((((h << (32 - bits)) | low) * INVERSE) & M32)).to_bytes(4, "little")


class Reject(Exception):
    pass


class Builder:
    def __init__(self, p, seed, window=None):
        self.p = p
        self.rnd = random.Random(seed)
        self.k = max(p.min_len, 2)
        self.win = window or p.max_dist
        self.b = bytearray()
        self.allowed = set()   # starts of k-grams that may repeat (inside copies)
        self.marked = set()    # positions of designed groups (and their copies)
        self.forbid = set()    # buckets that only designed groups may use
        self.grams = {}
        self.labels = {}
        self.group_heads = set()

    def _push(self, c):
        self.b.append(c)
        q = len(self.b) - self.k
        if q >= 0:
            self.grams[bytes(self.b[q:])] = q

    def _fits(self, c):
        q = len(self.b) - self.k + 1
        if q >= 0:
            last = self.grams.get(bytes(self.b[q:]) + bytes([c]))
            if last is not None and q - last <= self.win:
                return False
        if self.forbid and len(self.b) >= 3 and len(self.b) - 3 not in self.marked:
            v = int.from_bytes(bytes(self.b[-3:]) + bytes([c]), "little")
            if full_hash(v, self.p.hash_bits) & BUCKET_MASK in self.forbid:
                return False
        if self.forbid and len(self.b) >= 2 and self.p.hash_bits >= 32 - 24 + BUCKET_BITS and len(self.b) - 2 not in self.marked:
            # the bucket (product bits 32 - hash_bits ...) no longer depends on the group's 4th byte: decide it at the 3rd
            v = int.from_bytes(bytes(self.b[-2:]) + bytes([c]), "little")
            if full_hash(v, self.p.hash_bits) & BUCKET_MASK in self.forbid:
                return False
        return True

    def fresh(self, n):
        for _ in range(n):
            for _ in range(64):
                c = self.rnd.getrandbits(8)
                if self._fits(c):
                    break
            else:
                raise Reject("no fresh byte")
            self._push(c)

    def to_lane(self, lane, extra=0):
        """Fresh bytes until the next byte sits at `lane` of a 32-position step (at least `extra` of them)."""
        self.fresh(extra + (lane - len(self.b) - extra) % 32)

    def group(self, h):
        """Four bytes hashing to h, none equal to an earlier group's (only 2^(32 - hash_bits) groups share a hash value)."""
        g = group_with_hash(h, self.p.hash_bits, self.rnd)
        while g[:3] in self.group_heads:
            g = group_with_hash(h, self.p.hash_bits, self.rnd)
        self.group_heads.add(g[:3])
        self.marked.add(len(self.b))
        for c in g:
            self._push(c)

    def copy(self, src, length):
        """`length` bytes copied from position `src` (or a label): a planted match at distance len - src."""
        src = self.labels.get(src, src)
        start = len(self.b)
        for i in range(length):
            if src + i in self.marked:
                self.marked.add(start + i)
            self._push(self.b[src + i])
        self.allowed.update(range(start, start + length - self.k + 1))

    def label(self, name):
        self.labels[name] = len(self.b)

    def bytes(self):
        """The input, or Reject when a seam of a copy or a group made a repeat or a bucket use that was not planted."""
        b, k = bytes(self.b), self.k
        seen = {}
        for q in range(len(b) - k + 1):
            g = b[q:q + k]
            if g in seen and q - seen[g] <= self.win and q not in self.allowed:
                raise Reject(f"accidental {k}-gram repeat at {q}")
            seen[g] = q
        if self.forbid:
            for q in range(len(b) - 3):
                if q not in self.marked and full_hash(int.from_bytes(b[q:q + 4], "little"), self.p.hash_bits) & BUCKET_MASK in self.forbid:
                    raise Reject(f"a fresh position in a designed bucket at {q}")
        return b


def build_pair(p, seed, make, *variants, window=None):
    """`make(builder, variant)` for each variant from the same seed; retried with other seeds until both are clean."""
    for attempt in range(64):
        try:
            outs = []
            for v in variants:
                bd = Builder(p, seed * 1000 + attempt, window)
                make(bd, v)
                outs.append(bd.bytes())
            assert len({len(o) for o in outs}) == 1, "pair members differ in length"
            return outs
        except Reject:
            continue
    raise RuntimeError("no clean input in 64 seeds")


def _pick_hash(bd):
    h = bd.rnd.getrandbits(bd.p.hash_bits)
    bd.forbid.add(h & BUCKET_MASK)
    return h


# ---------------------------------------------------------------------------------------------------- flag-LZ finder profiles
def related(h, kind, bits):
    """Another hash value in h's bucket: `tag` differs in the three tag bits the node ring keeps, `tag3` agrees in them but not
    in the full value (only the re-hash tells), `collision` is h itself (different bytes, a real chain candidate)."""
    tag = h >> BUCKET_BITS
    if kind == "tag":
        return (h & BUCKET_MASK) | ((tag ^ 1) << BUCKET_BITS)
    if kind == "tag3":
        return (h & BUCKET_MASK) | ((tag ^ 8) << BUCKET_BITS)
    return h


def _decoys(p, seed, kinds_a, kinds_b, gap, split=False):
    """A real match (12 bytes) behind decoys of the same bucket; `split` puts half the decoys in front of a 40-byte gap (in the
    node ring) and half behind it (in the searching position's step)."""
    L = min(12, p.max_len)

    def make(bd, kinds):
        h = _pick_hash(bd)
        bd.fresh(48)
        bd.label("S")
        bd.group(h)
        bd.fresh(L + 4)
        half = len(kinds) // 2 if split else len(kinds)
        for i, kind in enumerate(kinds):
            if i == half:
                bd.fresh(40)
            if kind == "none":
                bd.fresh(6)
            else:
                bd.group(related(h, kind, p.hash_bits))
                bd.fresh(2)
        bd.fresh(gap)
        if p.min_table and p.min_len < 4:
            # from quality 10 a failed chain walk falls back to the latest position with the same first min_length bytes: give
            # it one that is not the real match
            bd.marked.add(len(bd.b))
            bd.copy("S", p.min_len)
            bd.fresh(3)
        bd.copy("S", L)
        bd.fresh(48)

    return build_pair(p, seed, make, kinds_a, kinds_b)


def profile_tags(p, seed):
    m = p.max_chain
    if m * 6 + 200 > WIN:
        return []
    out = []
    for gap in (0, 40):
        for kind in ("tag", "tag3"):
            a, b = _decoys(p, seed + gap, [kind] * m, ["collision"] * m, gap)
            out.append((f"{kind} x{m} / collision x{m}, gap {gap}", a, b))
    return out


def profile_chain(p, seed):
    """The winner is the max_chain-th or the (max_chain + 1)-th same-hash candidate; a tie goes to the nearer candidate."""
    m = p.max_chain
    if m * 6 + 240 > WIN:
        return []
    out = []
    for gap, split in ((0, False), (40, False), (0, True)):
        a, b = _decoys(p, seed + gap + split, ["collision"] * (m - 1) + ["none"], ["collision"] * m, gap, split)
        out.append((f"winner #{m} / #{m + 1}, gap {gap}{' split' if split else ''}", a, b))
    L = min(10, p.max_len - 1)

    def tie(bd, farther_longer):
        bd.fresh(40)
        bd.label("F")
        bd.fresh(L + 8)
        bd.copy("F", L)          # the nearer source agrees with the farther one on L bytes, then not
        bd.fresh(60)
        bd.copy("F", L + (1 if farther_longer else 0))   # the target: a tie, or one byte more from the farther source
        bd.fresh(40 if farther_longer else 41)

    if m >= 2:   # (with one attempt only the nearer candidate is compared)
        a, b = build_pair(p, seed, tie, False, True)
        out.append(("equal candidates / farther longer", a, b))
    return out


def profile_distance(p, seed, lanes=(0, 31), park=True):
    """The only candidate at max_dist - 1, max_dist or max_dist + 1; also right behind a parking pass of the heads."""
    L = min(12, p.max_len)
    D = p.max_dist
    out = []
    places = [(lane, 0) for lane in lanes] + ([(lane, PARK) for lane in (0, 31)] if park and D <= WIN else [])
    for lane, base in places:
        target = base + 64 + D + 32 + lane if base == 0 else base + lane

        def make(bd, d):
            h = _pick_hash(bd)
            bd.fresh(target - d)
            bd.label("S")
            bd.group(h)
            bd.fresh(d - 4)
            bd.copy("S", L)
            bd.fresh(48)

        for d0, d1 in ((D, D + 1), (D - 1, D + 1)):
            a, b = build_pair(p, seed + lane + base + d0, make, d0, d1)
            out.append((f"distance {d0} / {d1} at {target}", a, b))
    return out


def profile_lazy(p, seed):
    """A match of best_len at P and one of best_len + 1 (or equal, or long) at P + 1; P at lane 31 (the token stays pending
    across the step), 0 or 5."""
    T = p.lazy
    out = []
    if T + 3 > p.max_len or T < p.min_len:
        return out
    NL = min(40, p.max_len)   # (past the threshold there is no lazy test: the rest of the next match is a match of its own or not)
    for lane in (31, 0, 5):
        def make(bd, v):
            lk, nb = v   # the match at P and the one at P + 1
            bd.fresh(48)
            bd.label("A")
            bd.fresh(T + 8)
            bd.fresh(20)
            bd.label("B")
            bd.copy(bd.labels["A"] + 1, lk - 1)
            bd.fresh(NL + 10 - lk)
            bd.to_lane(lane, 16)
            P = len(bd.b)
            bd.copy("A", lk)
            bd.copy(bd.labels["B"] + lk - 1, nb - lk + 1)
            bd.allowed.update(range(P, P + nb + 1))
            if bd.b[bd.labels["A"] + lk] == bd.b[P + lk]:
                raise Reject("the match at P runs on")
            bd.fresh(NL + 4 - nb)
        for name, v0, v1 in (("next equal / longer", (T, T), (T, T + 1)), (f"best_len T + 1, next T + 2 / {NL}", (T + 1, T + 2), (T + 1, NL))):
            a, b = build_pair(p, seed + lane, make, v0, v1)
            out.append((f"lazy {name}, lane {lane}", a, b))
        if NL == 40 and lane == 31:
            a, b = build_pair(p, seed + 99, make, (T, T), (T, NL))
            out.append(("lazy next equal / covers the next step, lane 31", a, b))
    return out


def profile_long(p, seed):
    """Matches at and one byte past max_length, past the ring's lookahead (LZ11 family) and ending at the end of the stream."""
    if p.max_len <= LOOK:
        lengths = [(p.max_len - 1, p.max_len + 1)]   # (a match one byte past max_length is cut: the pair differs in the byte before)
    else:
        lengths = [(LOOK - 1, LOOK), (LOOK, LOOK + 1)]
    out = []
    for l0, l1 in lengths:
        for at_end in (False, True):
            def make(bd, L):
                bd.fresh(40)
                bd.label("S")
                bd.fresh(max(l0, l1) + 8)
                bd.to_lane(7)
                bd.copy("S", L)
                bd.fresh(max(l0, l1) - L + (0 if at_end else 40))
            a, b = build_pair(p, seed + l0, make, l0, l1)
            out.append((f"length {l0} / {l1}{' at the end' if at_end else ''}", a, b))
    return out


def profile_small(p, seed):
    """Quality >= 10 (small-match table, min_length < 4): the latest position with the same first min_length bytes is nearer
    than min_distance, so its distance is raised; once inside the buffer, once in front of position 0 (no match)."""
    if not (p.min_table and p.min_len < 4 and p.min_dist >= 2):
        return []
    out = []
    for lead in (1, 3):
        def make(bd, run):
            bd.fresh(lead)
            start = len(bd.b)
            for _ in range(run):
                bd._push(0)
            bd.allowed.update(range(start, start + run))
            bd.fresh(48 - run)
        a, b = build_pair(p, seed + lead, make, 4, 5 + p.min_dist - 2)
        out.append((f"raised distance, run after {lead}", a, b))
    return out


def head_at_start(n_run=4):
    """Streams that open with a run of zeros: at position 1 the raised small-match distance points in front of the buffer."""
    return [bytes(n_run) + bytes(range(1, 60)), bytes(n_run + 1) + bytes(range(7, 90))]


def profile_compat(p, seed):
    """CompatibilityMode: runs of period 1-4, whose match the reference cuts at its distance."""
    out = []
    for period in (1, 2, 3, 4):
        def make(bd, n):
            bd.fresh(40)
            start = len(bd.b)
            bd.fresh(period)
            for i in range(n - period):
                bd._push(bd.b[start + i])
            bd.allowed.update(range(start, start + n))
            bd.fresh(40 + 24 - n)
        a, b = build_pair(p, seed + period, make, 12, 24)
        out.append((f"period {period} run 12 / 24", a, b))
    return out


FLAG_PROFILES = {"tags": profile_tags, "chain": profile_chain, "distance": profile_distance, "lazy": profile_lazy,
                 "long": profile_long, "small": profile_small}


# ---------------------------------------------------------------------------------------------------- byte-LZ writer profiles
def profile_bytes(p, seed):
    fmt = p.fmt
    out = []

    def planted(name, v0, v1):
        """(lit, dist, length): a match of `length` bytes at `dist`, behind a literal run of `lit` bytes that an earlier 8-byte
        match closes; both members equally long, the target where it is in the other one, or one byte further."""
        D, Lmax = max(v0[1], v1[1]), max(v0[2], v1[2])

        def make(bd, v):
            lit, dist, length = v
            bd.fresh(24)
            bd.label("S")
            bd.group(_pick_hash(bd))   # no other position in its bucket: the planted source is the only candidate
            bd.fresh(length + 4)
            filler = dist - (length + 8) - 8 - lit
            if filler < 0:
                raise ValueError(f"{name}: no room for the closing match")
            bd.fresh(filler)
            bd.copy(0 if len(bd.b) + 8 < p.max_dist else len(bd.b) - 40, 8)
            bd.fresh(lit)
            bd.copy("S", length)
            bd.fresh(40 + D + Lmax - dist - length)
        a, b = build_pair(p, seed + len(out), make, v0, v1)
        out.append((name, a, b))

    # (a pair (e, e + 2) around an edge e where a token form gets one byte longer: e + 2 costs one byte more than e, e costs two
    #  literals more than e + 2; (e, e + 1) would cost the same)
    if fmt in (A.FMT_LZ4, A.FMT_LZ4_LEGACY, A.FMT_LZ4_BLOCK):
        planted("match 17 / 19", (6, 500, 17), (6, 500, 19))
        planted("match 272 / 274", (6, 600, 272), (6, 600, 274))
        planted("literals 14 / 15", (14, 500, 20), (15, 500, 20))
        planted("literals 269 / 270", (269, 900, 20), (270, 900, 20))
    elif fmt == A.FMT_LZO:
        planted("distance 0x800 / 0x801", (6, 0x800, 6), (6, 0x801, 6))
        planted("distance 0x4000 / 0x4001", (6, 0x4000, 20), (6, 0x4001, 20))
        planted("distance 0xBFFF / 0xC000", (6, 0xBFFF, 6), (6, 0xC000, 6))
        planted("length 8 / 10 near", (6, 300, 8), (6, 300, 10))
        planted("length 33 / 35", (6, 3000, 33), (6, 3000, 35))
        planted("length 9 / 11 far", (6, 0x5000, 9), (6, 0x5000, 11))
        planted("literals 3 / 4", (3, 300, 8), (4, 300, 8))
        planted("literals 18 / 19", (18, 300, 8), (19, 300, 8))
        planted("literals 273 / 274", (273, 900, 8), (274, 900, 8))
    elif fmt in (A.FMT_SNAPPY, A.FMT_SNAPPY_BLOCK):
        planted("literals 60 / 61", (60, 500, 8), (61, 500, 8))
        planted("literals 256 / 257", (256, 900, 8), (257, 900, 8))
        planted("copy length 11 / 13", (6, 500, 11), (6, 500, 13))
        planted("copy offset 2047 / 2048", (6, 2047, 8), (6, 2048, 8))
    elif fmt == A.FMT_PRS:
        planted("length 5 / 7", (6, 100, 5), (6, 100, 7))
        planted("length 9 / 11", (6, 1000, 9), (6, 1000, 11))
        planted("length 255 / 256", (6, 1000, 255), (6, 1000, 256))
    return out


def long_literal_runs():
    """Snappy literal runs of 65 536 bytes and more (tag 61 / 62), LZ4 / LZO runs past several length extensions."""
    rnd = random.Random(5)
    noise = bytes(rnd.getrandbits(8) for _ in range(70000))
    return [noise[:65536] + noise[:40], noise[:65537] + noise[:40], noise]


# ---------------------------------------------------------------------------------------------------- worst cases for the bound
def worst_cases(n, seed=3):
    """Inputs that make the token writers expand: noise; a far 3-byte match every 7 bytes (LZO M4 splits the literal run);
    2- and 3-byte matches every 4-5 bytes."""
    rnd = random.Random(seed)
    noise = bytearray(rnd.getrandbits(8) for _ in range(n))
    far = bytearray(noise)
    for q in range(0xC000 + 16, n - 3, 7):
        s = q - 0x4001 - rnd.randrange(0x7000)
        far[q:q + 3] = far[s:s + 3]
    short = bytearray(noise)
    q = 300
    while q < n - 3:
        L = 2 + (q & 1)
        s = q - 1 - rnd.randrange(250)
        short[q:q + L] = short[s:s + L]
        q += 4 + (q % 2)
    return {"noise": bytes(noise), "far3": bytes(far), "short": bytes(short)}
