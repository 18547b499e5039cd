// decode_flaglz.cu — batched decoder for the flag-byte LZ77 family: LZ10, LZ11, Yaz0/Yaz1, LZSS (interleaved
// flag/token streams) and MIO0, Yay0 (three separate sub-streams).  One compressed stream per warp.
//
// Reference semantics restated on the device (paths under /root/reference/src):
//   LZ10   AuroraLib.Compression.Nintendo/Nintendo/LZ10.cs:47-57 (header) :82-111 (body)
//   LZ11   .../Nintendo/LZ11.cs:43-53, :83-133
//   Yaz0   .../Nintendo/Yaz0.cs:58-79 (header + endian retry) -> Yay0.cs:110-144 (token core)
//   Yay0   .../Nintendo/Yay0.cs:50-60, :99-144
//   MIO0   .../Nintendo/MIO0.cs:51-61, :105-149
//   LZSS   AuroraLib.Compression/Formats/Common/LZSS.cs:53-69, :91-130
//   window AuroraLib.Compression/IO/LzWindows.cs:72-115 (BackCopy/OffsetCopy), FlagReader.cs:53-65
//
// Design (B200, sm_100a):
//   * persistent grid, ONE WARP PER STREAM SLOT, streams handed out by a global ticket (largest first when the host
//     supplies an order array); a block holds as many slots as its 227 KiB of shared memory allow;
//   * the compressed bytes are staged into a per-slot shared-memory ring by 1-D TMA bulk copies
//     (cp.async.bulk + mbarrier complete_tx), two 1 KiB chunks in flight per sub-stream;
//   * one flag GROUP per lane (256 tokens per warp iteration): the serial part is only the chain of group starts,
//     and runs of equally sized groups (all-literal, all-match) are resolved by one ballot instead of the walk;
//   * the decoded bytes live in a per-slot 8 KiB shared-memory ring that always holds the last 4 KiB window, so
//     back-references never touch HBM: literals are scattered lane-locally, the matches of an iteration are queued
//     and then resolved ONE MATCH PER LANE in dependency rounds (a match is ready when the last unresolved match
//     below it ends at or before its source), long matches warp-cooperatively, and the ring is drained to HBM in
//     512-byte, 16-byte-per-lane vector stores.
#include "common.cuh"
#include "stage.cuh"

namespace aurora {

namespace {

constexpr int kRing = 8192;          // per-slot output ring (bytes)
constexpr int kRingMask = kRing - 1;
constexpr int kWindow = 4096;        // largest back-reference distance of the family
constexpr int kSubMax = 2048;        // token-per-lane core: output bytes resolved per sub-batch
constexpr int kFlush = 512;          // bytes per ring->HBM drain step (16 B per lane)
#ifndef AURORA_HANDOFF_AT
#define AURORA_HANDOFF_AT 48
#endif
constexpr int kIterMatches = 144 - AURORA_HANDOFF_AT;    // match descriptors one iteration may queue (an iteration is cut at the group that would exceed it)
constexpr int kHandoffAt = AURORA_HANDOFF_AT;       // queued matches at which a batch is handed to the resolver warp
constexpr int kQueue = kIterMatches + kHandoffAt;   // entries of ONE queue buffer (a slot has two)
constexpr int kHandoffSpan = 2048;   // ... or this many bytes of literals
constexpr int kSubMaxG = 2304;       // smallest iteration budget the cores rely on (>= the largest single group: 8 x 273)
constexpr int kIterCap = kRing - kWindow;   // output bytes of one iteration: window + iteration fit the ring, and the
                                            // slots an iteration overwrites (positions 8192 lower) are below the window
                                            // and below everything not yet drained (< 512 bytes behind the iteration)
#ifndef AURORA_REG_DELTA
#define AURORA_REG_DELTA 16
#endif


enum Kind { K_LZ10 = 0, K_LZ11 = 1, K_YAZ0 = 2, K_LZSS = 3, K_MIO0 = 4, K_YAY0 = 5, K_HUDSON = 6, K_LZ40 = 7, K_SMSR = 8 };

// Shared memory of one stream slot (the launcher adds 8 KiB of alignment slack for the rings):
//   ring 8 KiB | staged sub-streams | match queue x2 | group offsets | mailboxes x2 + stream descriptor | TMA mbarriers
// A block holds kSlots slots served by 2 * kSlots warps (warpgroups alternate parser / resolver roles); a slot's parser and
// resolver hand batches over through two hardware named barriers, so kSlots <= 8 (16 barriers per block) and an SM runs
// as many blocks as its shared memory holds (two for the single-sub-stream formats).
template <int K>
struct Traits {
    static constexpr int kStreams = (K == K_MIO0 || K == K_YAY0) ? 3 : (K == K_SMSR) ? 2 : 1;
    static constexpr int kMaxTok = (K == K_LZ10 || K == K_MIO0 || K == K_SMSR) ? 18 : (K == K_YAZ0 || K == K_YAY0 || K == K_HUDSON) ? 273 : (K == K_LZSS) ? 258 : 65808;   // LZ11 65 808, LZ40 65 807
    static constexpr bool kNeedSub = kMaxTok * 32 > kSubMax;
    static constexpr int kQueueBytes = 2 * kQueue * 8;
    static constexpr int kAuxBytes = kStreams * kInStage + kQueueBytes + 128 + 48 + 2 * kStreams * 8;
    static constexpr int kSmemPerSlot = kRing + kAuxBytes;
#ifdef AURORA_FLAG_SLOTS
    static constexpr int kSlots = AURORA_FLAG_SLOTS;                      // developer probe: stream slots per block (4 or 8)
#else
    static constexpr int kSlots = 8 * kSmemPerSlot + kRing <= 115 * 1024 ? 8 : 4;
#endif
    static constexpr int kSmemPerBlock = kSlots * kSmemPerSlot + kRing;   // + alignment slack for the rings
    static constexpr int kBlocksPerSM = (228 * 1024) / (kSmemPerBlock + 1024) < 1 ? 1 : (228 * 1024) / (kSmemPerBlock + 1024);
    // registers: the launch gives every thread kLaunchRegs; the parser warpgroups then grow by kRegDelta and the resolver
    // warpgroups shrink by it (setmaxnreg; the sum stays in the block's pool)
    static constexpr int kLaunchRegs0 = (65536 / (kBlocksPerSM * kSlots * 64)) / 8 * 8;
    static constexpr int kLaunchRegs = kLaunchRegs0 > 128 ? 128 : kLaunchRegs0;
#ifdef AURORA_AFFINE
    static constexpr bool kRegSplit = false;
#else
    static constexpr bool kRegSplit = kLaunchRegs < 104;
#endif
    static constexpr int kParserRegs = kLaunchRegs + AURORA_REG_DELTA, kResolverRegs = kLaunchRegs - AURORA_REG_DELTA;
};

// out[dst+i] = out[dst-d + (i mod d)], i < len : LzWindows.BackCopy (IO/LzWindows.cs:72-100) on the flat ring.
// All reads are below dst and all writes at or above it, so one pass has no internal hazard.
__device__ __forceinline__ void ring_copy_match(uint8_t* ring, uint32_t dstp, uint32_t d, uint32_t len) {
    const uint32_t lane = lane_id();
    const uint32_t srcp = dstp - d;
    if (d >= len) {
        for (uint32_t i = lane; i < len; i += 32) ring[(dstp + i) & kRingMask] = ring[(srcp + i) & kRingMask];
    } else if (len < 512) {
        const uint32_t r = c_rcp.v[d];   // d < len < 512: uniform constant-bank load
        for (uint32_t i = lane; i < len; i += 32) {
            const uint32_t off = i - ((i * r) >> 20) * d;
            ring[(dstp + i) & kRingMask] = ring[(srcp + off) & kRingMask];
        }
    } else {
        for (uint32_t i = lane; i < len; i += 32) ring[(dstp + i) & kRingMask] = ring[(srcp + i % d) & kRingMask];
    }
}

struct OutState {
    uint8_t* ring;
    uint32_t rbase;    // shared address of the ring (8 KiB aligned)
    uint8_t* dst;
    uint32_t limit;    // bytes of the destination that may be written
    uint32_t flushed;  // output position drained to HBM so far (multiple of kFlush)
    bool aligned;
    // Chunks are retired as soon as they are produced, also past `limit` (overshooting tokens, destination smaller
    // than the output): bytes beyond the limit are dropped, but the bytes below it must leave the ring before a
    // long match wraps over them.
    __device__ __forceinline__ void drain(uint32_t produced) {
        const uint32_t lane = lane_id();
        while (flushed + kFlush <= produced) {
            if (aligned && flushed + kFlush <= limit) {
                const uint4 v = *reinterpret_cast<const uint4*>(ring + ((flushed + lane * 16) & kRingMask));
                *reinterpret_cast<uint4*>(dst + flushed + lane * 16) = v;
            } else if (flushed < limit) {
                for (uint32_t i = lane; i < kFlush; i += 32)
                    if (flushed + i < limit) dst[flushed + i] = ring[(flushed + i) & kRingMask];
            }
            flushed += kFlush;
        }
    }
    __device__ __forceinline__ void finish(uint32_t produced) {
        const uint32_t lane = lane_id();
        drain(produced);
        const uint32_t upto = min(produced, limit);
        for (uint32_t p = flushed + lane; p < upto; p += 32) dst[p] = ring[p & kRingMask];
    }
};

struct BodyResult {
    int status;
    uint32_t written;
    uint32_t consumed;
};

// ---------------------------------------------------------------------------------------------
// token core shared by all six formats.
//   interleaved formats: in[0] is the whole blob, cursor `cur` = blob offset of the next flag byte.
//   split formats: in[0] flags (relative to blob offset 0x10), in[1] codes (relative to comp_off),
//                  in[2] literals + extended lengths (relative to lit_off).
// ---------------------------------------------------------------------------------------------
template <int K>
__device__ BodyResult decode_body(InStream* in, OutState& out, const uint32_t slen, const uint32_t size,
                                  const uint32_t body_off, const uint32_t comp_off, const uint32_t lit_off,
                                  const LzssParams& lz) {
    const uint32_t lane = lane_id();
    const uint32_t lt_mask = (1u << lane) - 1u;
    uint8_t* ring = out.ring;
    uint32_t written = 0;
    uint32_t cur = (K == K_MIO0 || K == K_YAY0 || K == K_SMSR) ? 0u : body_off;
    uint32_t ccur = 0, lcur = 0;   // split formats: relative cursors
    uint32_t consumed = (K == K_MIO0 || K == K_YAY0) ? max(comp_off, lit_off) : (K == K_SMSR) ? lit_off : body_off;
    int status = AURORA_OK;

    while (written < size) {
        // ------------------------------------------------------------------ parse 32 tokens
        bool ism;            // match?
        uint32_t len;        // decoded bytes of this token
        uint32_t dist = 1;   // back-reference distance (LZSS: raw window offset until resolved below)
        uint32_t lit = 0;    // literal byte
        uint32_t tok_end = 0;// interleaved: blob offset just past the token
        bool bad;            // the token (or its flag byte) lies beyond the end of the input
        bool ext_used = false;   // Yay0: the token consumed an extended-length byte
        uint32_t next_cur;

        if constexpr (K == K_LZ10 || K == K_LZSS) {
            in[0].ensure(cur);
            // flag-byte chain: a group is 1 + 8 + (#matches) bytes.  m = match bits in wire bit order.
            const uint32_t p0 = cur;
            const uint32_t f0 = in[0].at(p0), m0 = (K == K_LZ10) ? f0 : (~f0 & 0xFFu);
            const uint32_t p1 = p0 + 9 + __popc(m0);
            const uint32_t f1 = in[0].at(p1), m1 = (K == K_LZ10) ? f1 : (~f1 & 0xFFu);
            const uint32_t p2 = p1 + 9 + __popc(m1);
            const uint32_t f2 = in[0].at(p2), m2 = (K == K_LZ10) ? f2 : (~f2 & 0xFFu);
            const uint32_t p3 = p2 + 9 + __popc(m2);
            const uint32_t f3 = in[0].at(p3), m3 = (K == K_LZ10) ? f3 : (~f3 & 0xFFu);
            next_cur = p3 + 9 + __popc(m3);
            const uint32_t g = lane >> 3, j = lane & 7;
            const uint32_t pg = g == 0 ? p0 : g == 1 ? p1 : g == 2 ? p2 : p3;
            const uint32_t mg = g == 0 ? m0 : g == 1 ? m1 : g == 2 ? m2 : m3;
            uint32_t before;
            if (K == K_LZ10) {   // MSB first (FlagReader bitOrder Big)
                ism = (mg >> (7 - j)) & 1;
                before = __popc(mg >> (8 - j));
            } else {             // LSB first
                ism = (mg >> j) & 1;
                before = __popc(mg & ((1u << j) - 1u));
            }
            const uint32_t tokoff = pg + 1 + j + before;
            const uint32_t b1 = in[0].at(tokoff), b2 = in[0].at(tokoff + 1);
            if (K == K_LZ10) {
                len = ism ? (b1 >> 4) + 3 : 1;
                dist = (((b1 & 0xF) << 8) | b2) + 1;
            } else {
                len = ism ? (b2 & ((1u << lz.length_bits) - 1u)) + uint32_t(lz.min_length) : 1;
                dist = ((b2 >> lz.length_bits) << 8) | b1;
            }
            lit = b1;
            tok_end = tokoff + (ism ? 2 : 1);
            bad = pg >= slen || tok_end > slen;
        } else if constexpr (K == K_YAZ0 || K == K_LZ11) {
            in[0].ensure(cur);
            uint32_t pg = cur, myoff = 0, mysz = 1, mypg = 0;
#pragma unroll
            for (int g = 0; g < 4; g++) {
                const uint32_t f = in[0].at(pg);
                const uint32_t hi = in[0].at(pg + 1 + lane) >> 4;
                const uint32_t e0 = __ballot_sync(kFull, hi == 0);
                const uint32_t e1 = (K == K_LZ11) ? __ballot_sync(kFull, hi == 1) : 0u;
                uint32_t off = 0;
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const uint32_t bit = (f >> (7 - i)) & 1;
                    const bool is_lit = (K == K_YAZ0) ? bit != 0 : bit == 0;
                    const uint32_t sz = is_lit ? 1u : 2u + ((e0 >> off) & 1u) + ((K == K_LZ11) ? 2u * ((e1 >> off) & 1u) : 0u);
                    if (lane == uint32_t(g * 8 + i)) {
                        myoff = pg + 1 + off;
                        mysz = sz;
                        mypg = pg;
                    }
                    off += sz;
                }
                pg += 1 + off;
            }
            next_cur = pg;
            ism = mysz >= 2;
            const uint32_t b1 = in[0].at(myoff), b2 = in[0].at(myoff + 1), b3 = in[0].at(myoff + 2);
            lit = b1;
            if (K == K_YAZ0) {
                dist = (((b1 & 0xF) << 8) | b2) + 1;
                // the extended length byte is read with Stream.ReadByte(): -1 at EOF -> 0x11 (Yay0.cs:131)
                const bool have_ext = myoff + 2 < slen;
                len = !ism ? 1 : (mysz == 3 ? (have_ext ? b3 + 0x12 : 0x11) : (b1 >> 4) + 2);
                tok_end = myoff + (ism ? 2 : 1);
                bad = mypg >= slen || tok_end > slen;
                if (mysz == 3 && have_ext) tok_end = myoff + 3;
            } else {
                const uint32_t b4 = in[0].at(myoff + 3);
                if (mysz == 3) {
                    dist = (((b2 & 0xF) << 8) | b3) + 1;
                    len = (((b1 & 0xF) << 4) | (b2 >> 4)) + 17;
                } else if (mysz == 4) {
                    dist = (((b3 & 0xF) << 8) | b4) + 1;
                    len = (((b1 & 0xF) << 12) | (b2 << 4) | (b3 >> 4)) + 273;
                } else {
                    dist = (((b1 & 0xF) << 8) | b2) + 1;
                    len = ism ? (b1 >> 4) + 1 : 1;
                }
                tok_end = myoff + mysz;
                bad = mypg >= slen || tok_end > slen;
            }
        } else if constexpr (K == K_SMSR) {
            // SMSR00.cs:91-134.  in[0] = the code section (relative to blob offset 0x10, comp_off = its addressable bytes), in[1] =
            // the literals (relative to lit_off).  A 16-bit big-endian mask word (MSB first, 1 = literal) is followed by the
            // 16-bit codes of its 0 bits, so the next mask sits 2 + 2 * zeros bytes further: two masks = the 32 tokens of
            // this iteration.  Code index -> popcount of 0 bits before, literal index -> popcount of 1 bits before.
            in[0].ensure(cur, 72);
            in[1].ensure(lcur, 40);
            const uint32_t m0 = (in[0].at(cur) << 8) | in[0].at(cur + 1);
            const uint32_t p1 = cur + 2 + 2 * (16 - __popc(m0));
            const uint32_t m1 = (in[0].at(p1) << 8) | in[0].at(p1 + 1);
            next_cur = p1 + 2 + 2 * (16 - __popc(m1));
            const uint32_t j = lane & 15;
            const uint32_t mk = lane < 16 ? m0 : m1, mpos = lane < 16 ? cur : p1;
            ism = ((mk >> (15 - j)) & 1u) == 0;
            const uint32_t lits_in = j ? __popc(mk >> (16 - j)) : 0;
            const uint32_t crel = mpos + 2 + 2 * (j - lits_in);
            const uint32_t lrel = lcur + lits_in + (lane < 16 ? 0u : uint32_t(__popc(m0)));
            const uint32_t b1 = in[0].at(crel), b2 = in[0].at(crel + 1);
            dist = (((b1 & 0xF) << 8) | b2) + 1;
            len = ism ? (b1 >> 4) + 3 : 1;
            lit = in[1].at(lrel);
            // the mask word and a code are span elements (IndexOutOfRange past the section), a literal is a ReadUInt8 of the stream
            bad = mpos + 2 > comp_off || (ism ? crel + 2 > comp_off : lit_off + lrel + 1 > slen);
        } else if constexpr (K == K_HUDSON) {
            // LZHudson.cs:54-55: FlagReader(source, Endian.Big, 4, Endian.Big) — one 4-byte big-endian flag word governs exactly
            // the 32 tokens of this iteration (bit 1 = literal, MSB first); tokens as Yaz0 (2 bytes, 3 when the high nibble
            // of the first byte is 0).  A token's size depends on its own first byte, so the 32 token starts are one uniform
            // walk over a ballot mask of "high nibble == 0" for the 96 bytes behind the flag word.
            in[0].ensure(cur);
            const uint32_t fw = (in[0].at(cur) << 24) | (in[0].at(cur + 1) << 16) | (in[0].at(cur + 2) << 8) | in[0].at(cur + 3);
            const uint32_t t0 = cur + 4;
            const uint64_t elo = uint64_t(__ballot_sync(kFull, (in[0].at(t0 + lane) >> 4) == 0)) |
                                 (uint64_t(__ballot_sync(kFull, (in[0].at(t0 + 32 + lane) >> 4) == 0)) << 32);
            const uint32_t ehi = __ballot_sync(kFull, (in[0].at(t0 + 64 + lane) >> 4) == 0);
            uint32_t off = 0, myoff = 0, mysz = 1;
#pragma unroll 4
            for (int i = 0; i < 32; i++) {
                const bool is_lit = ((fw >> (31 - i)) & 1u) != 0;
                const uint32_t eb = off < 64 ? uint32_t(elo >> off) & 1u : (ehi >> (off - 64)) & 1u;
                const uint32_t sz = is_lit ? 1u : 2u + eb;
                if (lane == uint32_t(i)) {
                    myoff = t0 + off;
                    mysz = sz;
                }
                off += sz;
            }
            next_cur = t0 + off;
            ism = mysz >= 2;
            const uint32_t b1 = in[0].at(myoff), b2 = in[0].at(myoff + 1), b3 = in[0].at(myoff + 2);
            lit = b1;
            dist = (((b1 & 0xF) << 8) | b2) + 1;
            const bool have_ext = myoff + 2 < slen;   // Stream.ReadByte() == -1 at EOF -> 0x11 (Yay0.cs:131)
            len = !ism ? 1 : (mysz == 3 ? (have_ext ? b3 + 0x12 : 0x11) : (b1 >> 4) + 2);
            tok_end = myoff + (ism ? 2 : 1);
            bad = cur + 4 > slen || tok_end > slen;   // the flag word is a ReadInt32: all four bytes or EndOfStream
            if (mysz == 3 && have_ext) tok_end = myoff + 3;
        } else {   // K_MIO0 / K_YAY0
            in[0].ensure(cur, 8);
            in[1].ensure(ccur, 72);
            in[2].ensure(lcur, 72);
            const uint32_t fw = (in[0].at(cur) << 24) | (in[0].at(cur + 1) << 16) | (in[0].at(cur + 2) << 8) | in[0].at(cur + 3);
            next_cur = cur + 4;
            ism = ((fw >> (31 - lane)) & 1) == 0;
            const uint32_t lits_before = lane ? __popc(fw >> (32 - lane)) : 0;
            const uint32_t m_before = lane - lits_before;
            const uint32_t crel = ccur + 2 * m_before;
            const uint32_t b1 = in[1].at(crel), b2 = in[1].at(crel + 1);
            dist = (((b1 & 0xF) << 8) | b2) + 1;
            uint32_t ext_before = 0;
            bool is_ext = false;
            if (K == K_YAY0) {
                is_ext = ism && (b1 >> 4) == 0;
                ext_before = __popc(__ballot_sync(kFull, is_ext) & lt_mask);
            }
            const uint32_t lrel = lcur + lits_before + ext_before;
            const uint32_t lb = in[2].at(lrel);
            lit = lb;
            const uint32_t fabs = 0x10 + cur + (lane >> 3), cabs = comp_off + crel, labs = lit_off + lrel;
            if (K == K_MIO0) {
                len = ism ? (b1 >> 4) + 3 : 1;
            } else {
                ext_used = is_ext && labs < slen;   // ReadByte() == -1 at EOF: nothing consumed, length 0x11
                len = !ism ? 1 : (is_ext ? (ext_used ? lb + 0x12 : 0x11) : (b1 >> 4) + 2);
            }
            bad = fabs >= slen || (ism ? cabs + 2 > slen : labs + 1 > slen);
        }

        // ------------------------------------------------------------------ output positions
        const uint32_t incl = warp_incl_scan(len);
        const uint32_t excl = incl - len;
        const uint32_t remaining = size - written;
        bool active = excl < remaining;
        const uint32_t badmask = __ballot_sync(kFull, active && bad);
        if (badmask) {
            const uint32_t first = __ffs(badmask) - 1;
            active = active && lane < first;
            status = AURORA_END_OF_STREAM;
        }
        const uint32_t amask = __ballot_sync(kFull, active);   // always a prefix of the lanes
        const uint32_t nact = __popc(amask);
        if (nact == 0) break;
        const uint32_t total = __shfl_sync(kFull, incl, nact - 1);
        const uint32_t pos = written + excl;   // output position of this token

        if constexpr (K == K_LZSS) {
            // LZSS.cs:122-126 + LzWindows.OffsetCopy (:108-115): absolute ring offset -> distance
            const uint32_t ring_len = 1u << lz.windows_bits;
            const uint32_t offset = (uint32_t(lz.max_distance) + dist - uint32_t(lz.windows_start)) & uint32_t(lz.max_distance - 1);
            const uint32_t rp = pos & (ring_len - 1);
            uint32_t d = rp >= offset ? rp - offset : rp - offset + ring_len;
            if (d == 0) d = ring_len;   // BackCopy(0, n) re-reads the slot it writes: the data one window back
            dist = d;
        }

        // source.Position after the last executed token
        if constexpr (K == K_MIO0 || K == K_YAY0) {
            ccur += 2 * __popc(__ballot_sync(kFull, active && ism));
            lcur += __popc(__ballot_sync(kFull, active && !ism)) + __popc(__ballot_sync(kFull, active && ext_used));
            consumed = max(comp_off + ccur, lit_off + lcur);
        } else if constexpr (K == K_SMSR) {
            lcur += __popc(__ballot_sync(kFull, active && !ism));
            consumed = lit_off + lcur;   // source.Position: behind the last literal read
        } else {
            consumed = __shfl_sync(kFull, tok_end, nact - 1);
        }
        cur = next_cur;

        // ------------------------------------------------------------------ copy phase (sub-batches of <= kSubMax bytes)
        uint32_t a = 0;
        while (a < nact) {
            uint32_t b = nact;
            if constexpr (Traits<K>::kNeedSub) {
                const uint32_t base_excl = __shfl_sync(kFull, excl, a);
                const uint32_t inm = __ballot_sync(kFull, active && lane >= a && incl - base_excl <= uint32_t(kSubMax));
                b = a + __popc(inm);
                if (b == a) {
                    // a single token longer than kSubMax (LZ11): periodic copy in segments
                    const uint32_t dstp = __shfl_sync(kFull, pos, a);
                    const uint32_t l = __shfl_sync(kFull, len, a);
                    const uint32_t d = __shfl_sync(kFull, dist, a);
                    for (uint32_t s = 0; s < l; s += kSubMax) {
                        const uint32_t seg = min(uint32_t(kSubMax), l - s);
                        ring_copy_match(ring, dstp + s, d, seg);
                        __syncwarp();
                        out.drain(dstp + s + seg);
                    }
                    a++;
                    continue;
                }
            }
            const bool mine = active && lane >= a && lane < b;
            if (mine && !ism) ring[pos & kRingMask] = uint8_t(lit);
            __syncwarp();
            uint32_t mm = __ballot_sync(kFull, mine && ism);
            while (mm) {
                const int k = __ffs(mm) - 1;
                mm &= mm - 1;
                const uint32_t dstp = __shfl_sync(kFull, pos, k);
                const uint32_t ld = __shfl_sync(kFull, len | (dist << 17), k);
                ring_copy_match(ring, dstp, ld >> 17, ld & 0x1FFFFu);
                __syncwarp();
            }
            out.drain(written + __shfl_sync(kFull, incl, b - 1));
            a = b;
        }
        written += total;
        if (status != AURORA_OK) break;
    }
    out.finish(written);
    if (status == AURORA_OK) {
        if (K == K_LZSS ? written != size : written > size) status = AURORA_SIZE_MISMATCH;
    }
    return BodyResult{status, written, consumed};
}


// one (long) match copied by the whole warp: out[pos + i] = out[pos - d + (i mod d)], i < len, on the 8 KiB aligned ring
// at shared address rb (LzWindows.BackCopy's chunk loop, IO/LzWindows.cs:72-100)
__device__ __forceinline__ void ring_copy_any(uint32_t rb, uint32_t pos, uint32_t d, uint32_t len) {
    const uint32_t lane = lane_id();
    const uint32_t srcp = pos - d;
    if (len <= 32) {
        if (lane < len) {
            uint32_t off = lane;
            if (d < len) off = lane - ((lane * c_rcp.v[d]) >> 20) * d;
            sts_u8(((pos + lane) & kRingMask) | rb, lds_u8(((srcp + off) & kRingMask) | rb));
        }
    } else if (d >= len) {
        for (uint32_t i = lane; i < len; i += 32) sts_u8(((pos + i) & kRingMask) | rb, lds_u8(((srcp + i) & kRingMask) | rb));
    } else if (len < 512 && d < 512) {
        const uint32_t r = c_rcp.v[d];
        for (uint32_t i = lane; i < len; i += 32) {
            const uint32_t off = i - ((i * r) >> 20) * d;
            sts_u8(((pos + i) & kRingMask) | rb, lds_u8(((srcp + off) & kRingMask) | rb));
        }
    } else {
        // long periodic run: i mod d kept incrementally (one division for the lane's start and one for the stride)
        uint32_t off = lane % d;
        const uint32_t step = 32 % d;
        for (uint32_t i = lane; i < len; i += 32) {
            sts_u8(((pos + i) & kRingMask) | rb, lds_u8(((srcp + off) & kRingMask) | rb));
            off += step;
            off -= off >= d ? d : 0u;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Match resolution (resolver warp).  The queue of a batch holds {pos, len | d << 17} in stream order; every literal of the
// batch is already in the ring.
//   run merging: encoders split a long run (or a 32-byte tile) into maximum-length matches with the same distance that
//   follow each other without a gap; such a chain is exactly one longer copy out[o] = out[o - d].  A lane-parallel pass
//   compacts every chain into one entry in place (chains are cut at 32-entry blocks);
//   replay: the merged entries run in stream order, a byte per lane and pass, two entries per step when the second one
//   does not read what the first one writes (both loads before both stores), the next pair prefetched with one 16-byte
//   load.  The merge pass already turns the common entry (<= 64 bytes, no ring wrap, not self-overlapping or a run of
//   period 1 / 2 / 4) into ready-made shared addresses, so a pair of them costs ~25 instructions instead of ~55.
// Measured and rejected in round 2 (profiles/r2_resolver_experiments.md): one entry per lane in dependency rounds — with a
// watermark readiness test and per-class copy routines (9-22 rounds per 32 entries), and with EXACT dependencies from two
// lane-parallel binary searches plus lane-local byte / word / 16-byte copies (tile sheets still need 8.4 rounds per 32
// entries: chains of picks of the same tile; 569 M instead of 627 M instructions but 373 instead of 456 GB/s) —,
// pointer-jumping of tile chains, in-order steps of up to four hazard-free matches on 8 lanes each, lane-parallel copies by
// the PARSER of the matches whose source is already final, a pattern-word path for long runs of period 1 / 2 / 4, and three
// queue buffers on polled shared-memory counters instead of the two named barriers (T +4 %, X -20 %).  The wide variants
// issue fewer instructions per match on paper; none beat this loop: the resolver is ONE warp bound by the latency of its
// dependent chain (entry -> addresses -> load -> store), dependency depth starves the rounds, and work moved to the
// parser competes for the same issue slots.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void resolve_matches(uint32_t rb, uint32_t qaddr, uint32_t nq) {
    const uint32_t lane = lane_id();
    if (nq == 0) return;
    const uint32_t lt = (1u << lane) - 1u;
    uint32_t nout = 0;
    for (uint32_t base = 0; base < nq; base += 32) {
        const uint32_t q = base + lane;
        const bool have = q < nq;
        uint2 e = make_uint2(0u, 0u);
        if (have) e = lds_u64(qaddr + 8 * q);
        const uint32_t px = __shfl_up_sync(kFull, e.x, 1), py = __shfl_up_sync(kFull, e.y, 1);
        const bool cont = have && lane > 0 && e.x == px + (py & 0x1FFFFu) && (e.y >> 17) == (py >> 17);
        const uint32_t heads = __ballot_sync(kFull, have && !cont);
        const uint32_t valid = __ballot_sync(kFull, have);
        // last entry of my chain: the lane before the next head (or the last valid lane of the block)
        const uint32_t after = heads & ~lt & ~(1u << lane);
        const uint32_t last = after ? uint32_t(__ffs(after) - 2) : uint32_t(31 - __clz(valid));
        const uint32_t tx = __shfl_sync(kFull, e.x, last & 31), ty = __shfl_sync(kFull, e.y, last & 31);
        __syncwarp();
        if (have && !cont) {
            const uint32_t ml = tx + (ty & 0x1FFFFu) - e.x, d = e.y >> 17;
            uint32_t ox = e.x, oy = ml | (e.y & 0xFFFE0000u);
            // SIMPLE entry (the common case): at most 64 bytes, not self-overlapping or a run with period 1 / 2 / 4, neither
            // range wraps the ring -> the replay loop gets ready-made shared addresses:
            //   x = destination address | len << 18 | source index mask << 25,  y = source address | 1 << 31
            const uint32_t da = e.x & kRingMask, sa = (e.x - d) & kRingMask;
            const bool periodic = d < ml;
            if (ml <= 64 && (!periodic || d == 1 || d == 2 || d == 4) && da + ml <= uint32_t(kRing) && sa + min(ml, d) <= uint32_t(kRing)) {
                ox = (da | rb) | (ml << 18) | ((periodic ? d - 1 : 127u) << 25);
                oy = (sa | rb) | 0x80000000u;
            }
            sts_u64(qaddr + 8 * (nout + __popc(heads & lt)), ox, oy);
        }
        nout += __popc(heads);
    }
    __syncwarp();
    // Two entries per step.  SIMPLE pairs (see the merge pass) take the short way: one byte per lane and half (lanes 0..31
    // copy bytes 0..31, then 32..63), both loads before both stores when the second entry does not read what the first one
    // writes; everything else goes through ring_copy_any.  The next pair is prefetched with one 16-byte load (the slots
    // past the end of the queue are readable: slack behind the queue); an odd count is padded with an empty SIMPLE entry.
    if (nout & 1u) {
        if (lane == 0) sts_u64(qaddr + 8 * nout, 0u, 0x80000000u);
        nout++;
        __syncwarp();
    }
    uint4 cur = lds_u128(qaddr);
#pragma unroll 1
    for (uint32_t q = 0; q < nout; q += 2) {
        const uint4 nx = lds_u128(qaddr + 8 * (q + 2));
        const uint32_t dst0 = cur.x & 0x3FFFFu, len0 = (cur.x >> 18) & 0x7Fu, pm0 = cur.x >> 25, src0 = cur.y & 0x3FFFFu;
        const uint32_t dst1 = cur.z & 0x3FFFFu, len1 = (cur.z >> 18) & 0x7Fu, pm1 = cur.z >> 25, src1 = cur.w & 0x3FFFFu;
        if (((cur.y & cur.w) >> 31) && (src1 + min(len1, pm1 + 1) <= dst0 || src1 >= dst0 + len0)) {
            uint32_t v0 = 0, v1 = 0;
            if (lane < len0) v0 = lds_u8(src0 + (lane & pm0));
            if (lane < len1) v1 = lds_u8(src1 + (lane & pm1));
            if (lane < len0) sts_u8(dst0 + lane, v0);
            if (lane < len1) sts_u8(dst1 + lane, v1);
            if (max(len0, len1) > 32) {
                const uint32_t l2 = lane + 32;
                if (l2 < len0) v0 = lds_u8(src0 + (l2 & pm0));
                if (l2 < len1) v1 = lds_u8(src1 + (l2 & pm1));
                if (l2 < len0) sts_u8(dst0 + l2, v0);
                if (l2 < len1) sts_u8(dst1 + l2, v1);
            }
            __syncwarp();
        } else {
#pragma unroll 1
            for (int h = 0; h < 2; h++) {
                const uint32_t x = h ? cur.z : cur.x, y = h ? cur.w : cur.y;
                if (y >> 31) {
                    const uint32_t dst = x & 0x3FFFFu, len = (x >> 18) & 0x7Fu, pm = x >> 25, src = y & 0x3FFFFu;
                    uint32_t v = 0, w = 0;
                    if (lane < len) v = lds_u8(src + (lane & pm));
                    if (lane + 32 < len) w = lds_u8(src + ((lane + 32) & pm));
                    if (lane < len) sts_u8(dst + lane, v);
                    if (lane + 32 < len) sts_u8(dst + lane + 32, w);
                } else {
                    ring_copy_any(rb, x, y >> 17, y & 0x1FFFFu);
                }
                __syncwarp();
            }
        }
        cur = nx;
    }
}

// one (possibly very long) match in segments of 2 KiB with a drain in between (LZ11: up to 65 808 bytes)
__device__ __forceinline__ void long_match_copy(OutState& out, uint32_t pos, uint32_t d, uint32_t len) {
    for (uint32_t sgm = 0; sgm < len; sgm += 2048) {
        const uint32_t seg = min(2048u, len - sgm);
        ring_copy_any(out.rbase, pos + sgm, d, seg);
        __syncwarp();
        out.drain(pos + sgm + seg);
    }
}

// ---------------------------------------------------------------------------------------------
// Parser / resolver pairs.  A stream slot is served by TWO warps.  The PARSER walks the token stream, scatters the literals
// into the slot's ring and queues the matches; when a batch is worth it (kHandoffAt matches or kHandoffSpan bytes) it
// hands the batch to the RESOLVER, which resolves the matches (resolve_matches) and drains the finished bytes to HBM while
// the parser works on the next batch.  Why two warps: the slot's shared memory (8 KiB window ring) bounds the STREAMS per
// SM to 16, and 16 warps leave the SM latency bound (measured: 50 % issue utilisation, stalls on fixed-latency
// dependencies); a second warp per stream doubles the instruction streams in flight without a second window.
//   hand-off: two queue buffers and two 16-byte mailboxes per slot, and two HARDWARE NAMED BARRIERS (bar.arrive / bar.sync
//   over the 64 threads of the pair): F "batch is there" (parser arrives, resolver syncs) and E "batch is done" (resolver
//   arrives, parser syncs).  The parser syncs on E before it hands the next batch over, so at most one batch is in
//   flight and each barrier sees exactly one arrive and one sync per batch; a waiting warp sleeps in the barrier unit and
//   issues nothing (round 1 polled mbarriers here: 30 % of all issued instructions).
//   ring safety: while the resolver works on batch A (positions [a, a + sA), sources >= a - 4096, undrained bytes
//   >= a - 511) the parser may write batch B up to position a + sA + sB; the slots it overwrites hold positions 8192
//   lower, so sA + sB <= kIterCap = 4096 keeps them below the window.
// (all members warp-uniform)
// ---------------------------------------------------------------------------------------------
enum : uint32_t { kMsgBegin = 1u, kMsgFinish = 2u, kMsgLong = 4u, kMsgExit = 8u };

#ifndef AURORA_SIMT   // (tests/simt models the two named barriers of a slot on its CPU lane emulation)
__device__ __forceinline__ void bar_sync(uint32_t id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void bar_arrive(uint32_t id) { asm volatile("bar.arrive %0, 64;" ::"r"(id) : "memory"); }
#endif

struct SlotSink {
    uint32_t rbase;        // shared address of the slot's ring
    uint32_t qbase;        // shared address of queue buffer 0 (buffer 1 follows kQueue entries later)
    uint32_t mail;         // shared address of mailbox 0 (mailbox 1 follows), then the stream descriptor
    uint32_t bar_f, bar_e; // named barriers of the slot
    uint32_t it;           // batches handed over in the lifetime of the warp
    uint32_t qn;           // matches queued in the current batch
    uint32_t start;        // first position of the current batch
    uint32_t produced;     // bytes scattered / queued so far
    uint32_t span_a;       // bytes of the batch in flight (0: none outstanding)
    bool outstanding;
    uint32_t flags_next;

    __device__ __forceinline__ void init() {
        it = qn = start = produced = span_a = flags_next = 0;
        outstanding = false;
    }
    // the batch in flight has been resolved and drained
    __device__ __forceinline__ void wait_idle() {
        if (outstanding) bar_sync(bar_e);
        outstanding = false;
        span_a = 0;
    }
    __device__ __forceinline__ void handoff(uint32_t flags, uint32_t x = 0) {
        wait_idle();
        __syncwarp();   // every lane's ring / queue stores are ordered before the arrive
        if (lane_id() == 0) sts_u128(mail + 16 * (it & 1), (flags & kMsgLong) ? x : qn, produced, flags | flags_next, 0u);
        __threadfence_block();
        bar_arrive(bar_f);
        it++;
        outstanding = true;
        span_a = produced - start;
        start = produced;
        qn = 0;
        flags_next = 0;
    }
    // new stream (or Yaz0's second attempt): the resolver is idle, so the ring and the descriptor are ours
    __device__ __forceinline__ void begin(uint8_t* ring, uint32_t fill, uint8_t* dst, uint32_t limit) {
        wait_idle();
        const uint32_t w = fill * 0x01010101u;
        const uint4 v = make_uint4(w, w, w, w);
        uint4* p = reinterpret_cast<uint4*>(ring + (kRing - kWindow));
        for (int i = lane_id(); i < kWindow / 16; i += 32) p[i] = v;
        if (lane_id() == 0) {
            const uint64_t a = reinterpret_cast<uint64_t>(dst);
            sts_u128(mail + 32, uint32_t(a), uint32_t(a >> 32), limit, (a & 15) == 0 ? 1u : 0u);
        }
        qn = start = produced = 0;
        flags_next = kMsgBegin;
        __syncwarp();
    }
    // output bytes the next iteration may produce
    __device__ __forceinline__ uint32_t cap() const { return uint32_t(kIterCap) - span_a - (produced - start); }
    // room for an iteration of up to `need` bytes behind what is queued: wait for the batch in flight, or hand the
    // current one over first; returns the shared address of the iteration's first queue entry
    __device__ __forceinline__ uint32_t acquire_deferred(uint32_t need) {
        need = min(need, uint32_t(kIterCap));
        if (need > cap()) {
            wait_idle();
            if (need > cap()) {
                handoff(0);
                if (need > cap()) wait_idle();
            }
        }
        return qbase + 8 * ((it & 1) * kQueue + qn);
    }
    __device__ __forceinline__ void submit_deferred(uint32_t nq, uint32_t produced_now) {
        qn += nq;
        produced = produced_now;
        if (qn >= uint32_t(kHandoffAt) || produced - start >= uint32_t(kHandoffSpan)) handoff(0);
    }
    // the cores that keep their own iteration budget: any cut they make must leave room for their largest group
    __device__ __forceinline__ uint32_t acquire() { return acquire_deferred(uint32_t(kSubMaxG)); }
    __device__ __forceinline__ void submit(uint32_t nq, uint32_t produced_now) { submit_deferred(nq, produced_now); }
    __device__ __forceinline__ void finish(uint32_t produced_now) {
        produced = produced_now;
        handoff(kMsgFinish);
    }
    // LZ11 long-group path: tokens one at a time
    __device__ __forceinline__ void single_literal(uint32_t pos, uint32_t b) {
        acquire_deferred(1);
        if (lane_id() == 0) sts_u8((pos & kRingMask) | rbase, b);
        produced = pos + 1;
    }
    __device__ __forceinline__ void long_match(uint32_t pos, uint32_t d, uint32_t len) {
        if (produced != start || qn) handoff(0);   // everything before the match
        wait_idle();
        if (lane_id() == 0) sts_u64(qbase + 8 * ((it & 1) * kQueue), pos, len | (d << 17));
        produced = pos + len;
        handoff(kMsgLong, 1);
        wait_idle();   // the match streams through the whole ring
    }
    __device__ __forceinline__ void exit() { handoff(kMsgExit); }
};

// resolver side: consumes batches until the parser says exit
__device__ void resolver_role(uint8_t* ring, uint32_t qbase, uint32_t mail, uint32_t bar_f, uint32_t bar_e) {
    OutState out;
    out.ring = ring;
    out.rbase = smem_u32(ring);
    out.dst = nullptr;
    out.limit = 0;
    out.flushed = 0;
    out.aligned = false;
    for (uint32_t m = 0;; m++) {
        const uint32_t b = m & 1;
        bar_sync(bar_f);
        const uint4 msg = lds_u128(mail + 16 * b);   // {nq, produced, flags, -}
        if (msg.z & kMsgExit) break;
        if (msg.z & kMsgBegin) {
            const uint4 d = lds_u128(mail + 32);
            out.dst = reinterpret_cast<uint8_t*>(uint64_t(d.x) | (uint64_t(d.y) << 32));
            out.limit = d.z;
            out.aligned = d.w != 0;
            out.flushed = 0;
        }
        const uint32_t q = qbase + 8 * b * kQueue;
        if (msg.z & kMsgLong) {
            const uint2 e = lds_u64(q);
            long_match_copy(out, e.x, e.y >> 17, e.y & 0x1FFFFu);
        } else {
#ifndef AURORA_EXP_NOREPLAY   // developer probe: parse-bound speed (output is wrong)
            if (msg.x) resolve_matches(out.rbase, q, msg.x);
#endif
        }
        if (msg.z & kMsgFinish) out.finish(msg.y);
        else out.drain(msg.y);
        __syncwarp();
        __threadfence_block();
        bar_arrive(bar_e);
    }
}

// ---------------------------------------------------------------------------------------------
// G32 token core for the fixed-token-size interleaved formats (LZ10, LZSS): one flag GROUP per lane, i.e. up to
// 256 tokens per warp iteration.  The only serial part is the chain of 32 group starts (p += 9 + popc(matches)); runs of
// equally sized groups (random data: all literals; runs, tiles: all matches) are resolved by one ballot: every lane
// looks at the flag byte its group would have if all groups before it had the size of the first one, and the walk starts
// behind the leading lanes that agree.  Every lane then sizes its own 8 tokens, one packed warp scan gives output bases
// and match-queue slots, and the tokens are placed in two passes: a branch-free TOKEN pass in which every lane scatters
// its literals and writes each match's position and token address into the match's own queue entry, and a MATCH pass in
// which ONE queued match per lane (32 per round, at most 3 rounds) decodes its token in place into the
// {pos, len | d << 17} that resolve_matches() reads.  All shared-memory traffic uses 32-bit shared addresses; the output
// ring is 8 KiB aligned, so the wrapped address (pos & mask) | base is a single LOP3.
// Before the split the match decode sat in a branch inside the per-slot loop; with ~10 % match tokens some lane of the
// warp holds a match at nearly every slot, so the warp issued both sides at all 8 slots (148 SASS instructions for the
// 8 slots of LZ10, now 50 for the token pass + 48 for the match pass).
// Measured and rejected: the match pass as a loop over its rounds (C2 596 GB/s against 611; mixed entropy 779 against 831:
// its run iterations queue 96 matches, and each round waited for its two dependent shared-memory loads before the next
// one started; the unrolled pass issues the loads of all rounds first).  Because the token pass already knows each match's
// queue entry, the match pass needs no lane -> (group, k-th match) mapping.  The mappings considered for it (an expand
// through the group-start table, __fns over a warp-wide match mask) were not built: on top of the group search each needs
// a segmented scan of the match lengths inside a group for the output position, which the token pass has in orel[].
// ---------------------------------------------------------------------------------------------
struct CutResult {
    uint32_t total, nq, nlan, consumed;
    bool eos;
};

// End of the output, end of the input, or an iteration over the byte budget whose first group does not fit: the tokens
// are cut one by one exactly where the reference stops (LZ10.cs:88-110 / LZSS.cs:100-126).  Out of line: it runs once or
// twice per stream and would only dilute the instruction cache of the hot loop; it re-reads the tokens from the staged
// window instead of taking the caller's register arrays.
template <int K>
__device__ __noinline__ CutResult g32_cut_tokens(uint32_t rb, uint32_t qaddr, uint32_t wa, uint32_t mya, uint32_t m, uint32_t written,
                                                 uint32_t gexcl, uint32_t gincl, uint32_t qexcl, uint32_t qincl, uint32_t remaining, uint32_t cap,
                                                 uint32_t cur, uint32_t slen, LzssParams lz) {
    const uint32_t lane = lane_id();
    const uint32_t lmask = (1u << lz.length_bits) - 1u;
    const bool taken = gexcl < remaining && gincl <= cap && qincl <= uint32_t(kIterMatches);
    const uint32_t lim = remaining - gexcl;   // only meaningful when taken
    const uint32_t gabs = cur + (mya - wa);   // blob offset of my flag byte
    uint32_t jexec = 0;
    bool eos_here = false;
    {
        uint32_t a = gabs + 1, sa = mya + 1, o = 0;
        bool stop = false;
#pragma unroll 1
        for (int j = 0; j < 8; j++) {
            const bool ism = (K == K_LZ10) ? (m >> (7 - j)) & 1 : (m >> j) & 1;
            uint32_t len = 1;
            if (ism) len = (K == K_LZ10) ? (lds_u8(sa) >> 4) + 3 : (lds_u8(sa + 1) & lmask) + uint32_t(lz.min_length);
            const uint32_t tend = a + (ism ? 2 : 1);
            const bool want = o < lim;
            const bool bad = gabs >= slen || tend > slen;
            if (!stop && want && bad) eos_here = true;
            stop = stop || !want || bad;
            if (!stop) jexec = j + 1;
            a = tend;
            sa += ism ? 2 : 1;
            o += len;
        }
    }
    if (!taken) {
        jexec = 0;
        eos_here = false;
    }
    CutResult r{0u, 0u, 0u, 0u, false};
    const uint32_t eosmask = __ballot_sync(kFull, eos_here);
    if (eosmask) {
        const uint32_t gb = __ffs(eosmask) - 1;
        if (lane > gb) jexec = 0;
        r.eos = true;
    }
    r.nlan = __popc(__ballot_sync(kFull, jexec > 0));   // a prefix of the lanes
    if (r.nlan == 0) return r;
    const uint32_t last = r.nlan - 1;
    uint32_t oend = 0, qi = qexcl, aend = 0;
    {
        uint32_t sa = mya + 1, o = 0;
#pragma unroll 1
        for (int j = 0; j < 8; j++) {
            const bool ism = (K == K_LZ10) ? (m >> (7 - j)) & 1 : (m >> j) & 1;
            const bool e = uint32_t(j) < jexec;
            const uint32_t pos = written + gexcl + o;
            const uint32_t b1 = lds_u8(sa);
            uint32_t len = 1;
            if (e && !ism) sts_u8((pos & kRingMask) | rb, b1);
            if (ism) {
                const uint32_t b2 = lds_u8(sa + 1);
                uint32_t dist;
                if (K == K_LZ10) {
                    len = (b1 >> 4) + 3;
                    dist = (((b1 & 0xF) << 8) | b2) + 1;
                } else {
                    len = (b2 & lmask) + uint32_t(lz.min_length);
                    const uint32_t raw = ((b2 >> lz.length_bits) << 8) | b1;
                    const uint32_t ring_len = 1u << lz.windows_bits;
                    const uint32_t offset = (uint32_t(lz.max_distance) + raw - uint32_t(lz.windows_start)) & uint32_t(lz.max_distance - 1);
                    const uint32_t rp = pos & (ring_len - 1);
                    dist = rp >= offset ? rp - offset : rp - offset + ring_len;
                    if (dist == 0) dist = ring_len;
                }
                if (e) {
                    sts_u64(qaddr + 8 * qi, pos, len | (dist << 17));
                    qi++;
                }
            }
            sa += ism ? 2 : 1;
            o += len;
            if (e) {
                oend = o;
                aend = sa - wa;
            }
        }
    }
    r.total = __shfl_sync(kFull, gexcl + oend, last);
    r.nq = __shfl_sync(kFull, qi, last);
    r.consumed = cur + __shfl_sync(kFull, aend, last);
    return r;
}

template <int K, class Sink>
__device__ BodyResult decode_body_g32(InStream* in, Sink& sink, const uint32_t gaddr, const uint32_t slen,
                                      const uint32_t size, const uint32_t body_off, const LzssParams& lz) {
    const uint32_t lane = lane_id();
    const uint32_t rb = sink.rbase;
    uint32_t written = 0, cur = body_off, consumed = body_off;
    int status = AURORA_OK;
    const uint32_t lmask = (1u << lz.length_bits) - 1u;
    auto mbits = [](uint32_t fb) { return K == K_LZ10 ? fb : (fb ^ 0xFFu); };   // flag byte -> match bits in wire bit order

    while (written < size) {
        in[0].ensure(cur, kInMirror - 16);
        const uint32_t wa = smem_u32(in[0].window(cur));
        const uint32_t remaining = size - written;
        // ---- chain of 32 group starts; bounded by 32 * 17 = 544 < kInMirror for any data
        uint32_t mya, chain_end;
        {
            const uint32_t s = 9 + __popc(mbits(lds_u8(wa)));       // size of the first group
            mya = wa + lane * s;                                       // my group's start if all groups before it have that size
            const uint32_t nok = ~__ballot_sync(kFull, 9 + __popc(mbits(lds_u8(mya))) == s);
            if (nok == 0) {
                chain_end = 32 * s;
                if (s == 9 && remaining >= 256 && cur + 288 <= slen) {
                    // ---- 32 all-literal groups: 256 bytes, lane g copies in[9 g + 1 .. 9 g + 8] to out[8 g .. 8 g + 7]
                    sink.acquire_deferred(256);
                    const uint32_t t = written + 8 * lane;
                    if ((written & kRingMask) <= uint32_t(kRing - 256)) {
                        const uint32_t ta = (t & kRingMask) | rb;
#pragma unroll
                        for (int j = 0; j < 8; j++) sts_u8(ta + j, lds_u8(mya + 1 + j));
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; j++) sts_u8(((t + j) & kRingMask) | rb, lds_u8(mya + 1 + j));
                    }
                    written += 256;
                    cur += 288;
                    consumed = cur;
                    sink.submit_deferred(0, written);
                    continue;
                }
            } else {
                uint32_t k = __ffs(nok) - 1;   // >= 1: groups 0..k start where the guess says; go on from group k
                uint32_t ca = wa + k * s;
                chain_end = 0;
                // (Measured and rejected, round 2: guessing that the groups behind group k are all-literal — 80 % of the C2
                //  corpus's groups are — and finding the first lane that is not with one ballot per round.  ~12 instructions and
                //  two dependent shared-memory loads per round against 4 instructions per group here: 508 vs 545 GB/s.)
                if (chain_end == 0) {
#define AURORA_CHAIN_STEP(g)                                   \
    case g:                                                    \
        sts_u32(gaddr + 4 * g, ca);                            \
        ca += 9 + __popc(mbits(lds_u8(ca)));
                switch (k) {
                    AURORA_CHAIN_STEP(1) AURORA_CHAIN_STEP(2) AURORA_CHAIN_STEP(3) AURORA_CHAIN_STEP(4) AURORA_CHAIN_STEP(5)
                    AURORA_CHAIN_STEP(6) AURORA_CHAIN_STEP(7) AURORA_CHAIN_STEP(8) AURORA_CHAIN_STEP(9) AURORA_CHAIN_STEP(10)
                    AURORA_CHAIN_STEP(11) AURORA_CHAIN_STEP(12) AURORA_CHAIN_STEP(13) AURORA_CHAIN_STEP(14) AURORA_CHAIN_STEP(15)
                    AURORA_CHAIN_STEP(16) AURORA_CHAIN_STEP(17) AURORA_CHAIN_STEP(18) AURORA_CHAIN_STEP(19) AURORA_CHAIN_STEP(20)
                    AURORA_CHAIN_STEP(21) AURORA_CHAIN_STEP(22) AURORA_CHAIN_STEP(23) AURORA_CHAIN_STEP(24) AURORA_CHAIN_STEP(25)
                    AURORA_CHAIN_STEP(26) AURORA_CHAIN_STEP(27) AURORA_CHAIN_STEP(28) AURORA_CHAIN_STEP(29) AURORA_CHAIN_STEP(30)
                    AURORA_CHAIN_STEP(31)
                    default: break;
                }
#undef AURORA_CHAIN_STEP
                chain_end = ca - wa;
                __syncwarp();
                if (lane > k) mya = lds_u32(gaddr + 4 * lane);
                __syncwarp();   // the table is rewritten by the next iteration's walk
                }
            }
        }
        const uint32_t myrel = mya - wa;
        const uint32_t m = mbits(lds_u8(mya));   // match bits in wire bit order

        // ---- pass 1: sizes of my 8 tokens; tv[j] = shared address of token j << 8 | its first byte (shared addresses are
        //      below 2^24, and the literal store takes the low byte)
        uint32_t tv[8], orel[8];
        uint32_t gsize = 0;
        {
            uint32_t a = mya + 1;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const bool ism = (K == K_LZ10) ? (m >> (7 - j)) & 1 : (m >> j) & 1;
                const uint32_t b1 = lds_u8(a);
                tv[j] = (a << 8) | b1;
                orel[j] = gsize;
                uint32_t len;
                if (K == K_LZ10) len = ism ? (b1 >> 4) + 3 : 1;
                else len = ism ? (lds_u8(a + 1) & lmask) + uint32_t(lz.min_length) : 1;
                gsize += len;
                a += ism ? 2 : 1;
            }
        }
        const uint32_t nm = __popc(m);
        const uint32_t incl = warp_incl_scan(gsize | (nm << 20));
        const uint32_t gincl = incl & 0xFFFFFu, gexcl = gincl - gsize;
        const uint32_t qexcl = (incl >> 20) - nm;
        const uint32_t gbase = written + gexcl;
        uint32_t total, nq, nlan;
        // matches may stay queued across iterations (SlotSink): room for this iteration, or resolve first
        const uint32_t qaddr = sink.acquire_deferred(__shfl_sync(kFull, incl, 31) & 0xFFFFFu);
        const uint32_t cap = sink.cap();
        // groups that fit the byte budget and the queue (a prefix of the lanes): all of their tokens execute unless the
        // output or the input ends inside them
        const uint32_t nl = __popc(__ballot_sync(kFull, gincl <= cap && (incl >> 20) <= uint32_t(kIterMatches)));
        const uint32_t cut = __shfl_sync(kFull, incl, (nl + 31) & 31);
        const uint32_t end_rel = nl == 32 ? chain_end : __shfl_sync(kFull, myrel, nl & 31);
        if (nl > 0 && (cut & 0xFFFFFu) <= remaining && cur + end_rel <= slen) {
            // ---- fast path: every token of the first nl groups executes.  Token pass: a literal stores its byte, a match
            //      stores {pos, tv} into its queue entry; both stores are predicated, nothing branches per slot
            if (lane < nl) {
                uint32_t qa = qaddr + 8 * qexcl;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const bool ism = (K == K_LZ10) ? (m >> (7 - j)) & 1 : (m >> j) & 1;
                    const uint32_t pos = gbase + orel[j];
                    if (!ism) sts_u8((pos & kRingMask) | rb, tv[j]);
                    if (ism) {
                        sts_u64(qa, pos, tv[j]);
                        qa += 8;
                    }
                }
            }
            total = cut & 0xFFFFFu;
            nq = cut >> 20;
            __syncwarp();
            // ---- match pass: ONE queued match per lane decodes its token in place into {pos, len | dist << 17}
            {
                // the loads of all rounds are issued before their first use
                constexpr int kRounds = (kIterMatches + 31) / 32;
                uint32_t wv[kRounds], b2v[kRounds];
#pragma unroll
                for (int r = 0; r < kRounds; r++)
                    if (lane + 32 * r < nq) wv[r] = lds_u32(qaddr + 8 * (lane + 32 * r) + 4);
#pragma unroll
                for (int r = 0; r < kRounds; r++)
                    if (lane + 32 * r < nq) b2v[r] = lds_u8((wv[r] >> 8) + 1);
#pragma unroll
                for (int r = 0; r < kRounds; r++) {
                    if (lane + 32 * r < nq) {
                        const uint32_t e = qaddr + 8 * (lane + 32 * r), w = wv[r], b1 = w & 0xFFu, b2 = b2v[r];
                        uint32_t len, dist;
                        if (K == K_LZ10) {
                            len = (b1 >> 4) + 3;
                            dist = (((b1 & 0xF) << 8) | b2) + 1;
                        } else {
                            len = (b2 & lmask) + uint32_t(lz.min_length);
                            const uint32_t raw = ((b2 >> lz.length_bits) << 8) | b1;
                            const uint32_t ring_len = 1u << lz.windows_bits;
                            const uint32_t offset = (uint32_t(lz.max_distance) + raw - uint32_t(lz.windows_start)) & uint32_t(lz.max_distance - 1);
                            const uint32_t rp = lds_u32(e) & (ring_len - 1);
                            dist = rp >= offset ? rp - offset : rp - offset + ring_len;
                            if (dist == 0) dist = ring_len;
                        }
                        sts_u32(e + 4, len | (dist << 17));
                    }
                }
            }
            nlan = nl;
            consumed = cur + end_rel;
        } else {
            const CutResult r = g32_cut_tokens<K>(rb, qaddr, wa, mya, m, written, gexcl, gincl, qexcl, incl >> 20, remaining, cap, cur, slen, lz);
            if (r.eos) status = AURORA_END_OF_STREAM;
            if (r.nlan == 0) break;
            total = r.total;
            nq = r.nq;
            nlan = r.nlan;
            consumed = r.consumed;
        }
        written += total;
        sink.submit_deferred(nq, written);
        if (status != AURORA_OK) break;
        cur += (nlan == 32) ? chain_end : __shfl_sync(kFull, myrel, nlan & 31);
    }
    sink.finish(written);
    if (status == AURORA_OK) {
        if (K == K_LZSS ? written != size : written > size) status = AURORA_SIZE_MISMATCH;
    }
    return BodyResult{status, written, consumed};
}

// ---------------------------------------------------------------------------------------------
// G32 core for Yaz0/Yaz1 (Yay0.cs:110-144 through Yaz0.cs:91-92), LZ11 (LZ11.cs:83-133) and LZ40 / LZ60 (LZ40.cs:73-124: the flag
// byte is negated, a match is a little-endian u16 DDDDDDDD DDDDLLLL whose LOW nibble selects the size, distance 0 is one
// window back).  A match token is 2 bytes, or 3
// when the selector nibble of its first byte is 0 (LZ11 / LZ40: also 4 when it is 1), so a group's size depends on its own data and the chain of group starts cannot be a pure
// popcount chain.  The chain is still the only serial part: per group the warp loads the flag byte, builds a ballot mask
// E of "high nibble == 0" over the group's next 32 bytes, and walks only the MATCH tokens of the group (highest flag bit
// first) accumulating the number of 3-byte tokens: token i starts at 1 + i + matches_before + ext_before, and its
// ext bit is E[that offset - 1].  About 14 + 11 * matches instructions per group; everything else is lane-parallel.
// (A fixed-point iteration over guessed group starts was tried first; on data with many long matches it needs one
// round per group and was slower.)
// ---------------------------------------------------------------------------------------------
template <int K, class Sink>   // K_YAZ0, K_LZ11 or K_LZ40
__device__ BodyResult decode_body_g32_var(InStream* in, Sink& sink, const uint32_t gaddr, const uint32_t slen,
                                           const uint32_t size, const uint32_t body_off) {
    const uint32_t lane = lane_id();
    const uint32_t rb = sink.rbase;
    uint32_t written = 0, cur = body_off, consumed = body_off;
    int status = AURORA_OK;
    constexpr bool kFour = K == K_LZ11 || K == K_LZ40;                 // 2/3/4-byte match tokens (Yaz0: 2/3)
    // the nibble of a match token's first byte that selects its size (0 -> 3 bytes, 1 -> 4 bytes): LZ40 keeps the length in
    // the LOW nibble of a little-endian u16 (LZ40.cs:98-113), the others in the high nibble of the first byte
    auto sel = [](uint32_t b1) { return K == K_LZ40 ? (b1 & 0xFu) : (b1 >> 4); };
    // flag byte -> "bit set = match" (MSB first): Yaz0 inverts, LZ40 negates ((byte)-ReadByte(), LZ40.cs:88)
    auto mbits = [](uint32_t fb) { return K == K_YAZ0 ? (fb ^ 0xFFu) : K == K_LZ40 ? ((0u - fb) & 0xFFu) : fb; };
    // Chain reuse: an iteration cut by the byte budget executes only its first groups; the starts of the others stay
    // exact, so they are carried (as offsets relative to the next window) instead of being walked again.
    uint32_t nkeep = 0, chain_rel = 0;   // carried groups; offset at which the walk continues

    while (written < size) {
        in[0].ensure(cur, kInMirror - 16);
        const uint32_t wa = smem_u32(in[0].window(cur));
        const uint32_t wlimit = kInMirror - 48;   // a group may start in the first 592 bytes of the window (it is <= 33 bytes)
        // ---- 32 all-literal groups (random / incompressible stretches): 256 bytes, lane g copies in[9 g + 1 .. 9 g + 8] to
        //      out[8 g .. 8 g + 7] — the same fast path as the fixed-token core (round 2: Yaz0 on mixed-entropy data 342 -> see
        //      profiles/r2_probe_all_formats.log)
        if (nkeep == 0 && chain_rel == 0 && size - written >= 256 && cur + 288 <= slen) {
            const uint32_t ga = wa + 9 * lane;
            if (__all_sync(kFull, mbits(lds_u8(ga)) == 0)) {
                sink.acquire_deferred(256);
                const uint32_t t = written + 8 * lane;
                if ((written & kRingMask) <= uint32_t(kRing - 256)) {
                    const uint32_t ta = (t & kRingMask) | rb;
#pragma unroll
                    for (int j = 0; j < 8; j++) sts_u8(ta + j, lds_u8(ga + 1 + j));
                } else {
#pragma unroll
                    for (int j = 0; j < 8; j++) sts_u8(((t + j) & kRingMask) | rb, lds_u8(ga + 1 + j));
                }
                written += 256;
                cur += 288;
                consumed = cur;
                sink.submit_deferred(0, written);
                continue;
            }
        }
        // ---- exact chain of group starts (offsets relative to the window)
        uint32_t nvalid;
        {
            const uint32_t rel = lane < nkeep ? lds_u32(gaddr + 4 * lane) : 0xFFFFFFFFu;
            nvalid = __popc(__ballot_sync(kFull, rel <= wlimit));       // carried groups that start inside this window (a prefix)
            if (nvalid < nkeep) chain_rel = __shfl_sync(kFull, rel, nvalid);
        }
        uint32_t ca = wa + chain_rel;
#pragma unroll 1
        for (uint32_t g = nvalid; g < 32; g++) {
            if (ca - wa > wlimit) break;
            const uint32_t fb = lds_u8(ca);
            uint32_t mm = mbits(fb), x = 0, cnt = 0;                                       // match bits, MSB first
#ifndef AURORA_NO_LITRUN
            if (mm == 0) {
                // All-literal groups (9 bytes, ~80 % of the groups of asset data) come in runs: lane i looks at the flag byte
                // group g + i has if the run reaches it, one ballot measures the run and all of its starts are stored at once
                // (a step of this walk costs ~14 instructions per group).
                const uint32_t sa = ca + 9 * lane;
                const bool lit = sa - wa <= wlimit && lane < 32 - g && mbits(lds_u8(sa)) == 0;
                const uint32_t lm = __ballot_sync(kFull, lit);
                const uint32_t run = lm == 0xFFFFFFFFu ? 32u : uint32_t(__ffs(int(~lm))) - 1u;   // >= 1: lane 0 is this group
                if (lane < run) sts_u32(gaddr + 4 * (g + lane), sa - wa);
                ca += 9 * run;
                g += run - 1;
                nvalid = g + 1;
                continue;
            }
#endif
            sts_u32(gaddr + 4 * g, ca - wa);
            const uint32_t hi4 = sel(lds_u8(ca + 1 + lane));
            if (mm) {   // an all-literal group is 9 bytes: no extension masks, no walk
                const uint32_t E = __ballot_sync(kFull, hi4 == 0);                         // +1 byte
                const uint32_t E2 = kFour ? __ballot_sync(kFull, hi4 == 1) : 0u;           // +2 bytes (LZ11 / LZ40 4-byte tokens)
                // (Measured and rejected, round 1: skipping the walk when no candidate first byte of a match token — a 256-entry
                //  table of positions "if nothing is extended" ANDed with E | E2 — selects an extended token: Yaz0 275 vs 275,
                //  LZ11 180 vs 187, LZ40 219 vs 221 GB/s on the C2 corpus; the chain is not what bounds the parser.)
                do {   // visit only the match tokens (a branch-free walk over all eight tokens was measured: no gain)
                    const uint32_t hb = 31 - __clz(mm);
                    const uint32_t at = 7 - hb + cnt + x;
                    x += ((E >> at) & 1u) + 2u * ((E2 >> at) & 1u);
                    cnt++;
                    mm ^= 1u << hb;
                } while (mm);
            }
            ca += 9 + cnt + x;
            nvalid = g + 1;
        }
        __syncwarp();
        const bool valid = lane < nvalid;
        const uint32_t myrel = valid ? lds_u32(gaddr + 4 * lane) : 0u;
        const uint32_t mya = wa + myrel;

        // ---- pass 1: my 8 tokens
        uint32_t b1v[8], lenv[8], orel[8];
        uint32_t gsize = 0, gin;
        const uint32_t f = mbits(lds_u8(mya));   // bit set = match
        {
            uint32_t a = mya + 1;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const bool lit = ((f >> (7 - j)) & 1) == 0;
                const uint32_t b1 = lds_u8(a);
                const uint32_t n = sel(b1);
                b1v[j] = b1;
                orel[j] = gsize;
                if (K == K_YAZ0) {
                    const bool ext = !lit && n == 0;
                    const uint32_t b3 = lds_u8(a + 2);
                    lenv[j] = lit ? 1u : (ext ? b3 + 0x12u : n + 2u);
                    a += lit ? 1u : (ext ? 3u : 2u);
                } else if (K == K_LZ40) {
                    const uint32_t b3 = lds_u8(a + 2), b4 = lds_u8(a + 3);
                    uint32_t l = n, sz = 2;   // DDDDDDDD DDDDLLLL little-endian: lengths 2..15 in the nibble itself
                    if (n == 0) { l = b3 + 16; sz = 3; }
                    if (n == 1) { l = (b3 | (b4 << 8)) + 272; sz = 4; }
                    lenv[j] = lit ? 1u : l;
                    a += lit ? 1u : sz;
                } else {
                    const uint32_t b2 = lds_u8(a + 1), b3 = lds_u8(a + 2);
                    uint32_t l = n + 1, sz = 2;
                    if (n == 0) { l = (((b1 & 0xF) << 4) | (b2 >> 4)) + 17; sz = 3; }
                    if (n == 1) { l = (((b1 & 0xF) << 12) | (b2 << 4) | (b3 >> 4)) + 273; sz = 4; }
                    lenv[j] = lit ? 1u : l;
                    a += lit ? 1u : sz;
                }
                gsize += lenv[j];
            }
            gin = a - mya;
        }
        const uint32_t nm = __popc(f);
        const uint32_t gclamp = min(gsize, 8191u);   // LZ11 groups can be huge; anything above the iteration budget takes the long-group path
        const uint32_t incl = warp_incl_scan(valid ? (gclamp | (nm << 20)) : 0u);
        const uint32_t gincl = incl & 0xFFFFFu, gexcl = gincl - (valid ? gclamp : 0u);
        const uint32_t qexcl = (incl >> 20) - (valid ? nm : 0u);
        const uint32_t remaining = size - written;
        const uint32_t gbase = written + gexcl;
        const uint32_t qaddr = sink.acquire();   // the first ring / queue store of the iteration is below
        uint32_t jexec, nlan;
      for (;;) {
        // ---- which of my tokens execute (end of output, end of input, iteration byte budget, queue capacity)
        const uint32_t cap = sink.cap();
        const bool taken = valid && gexcl < remaining && gincl <= cap && (incl >> 20) <= uint32_t(kIterMatches);
        const uint32_t lim = remaining - gexcl;
        jexec = 8;
        bool eos_here = false;
        // fast path: every token of every valid group executes (not the end of the output, all input bytes present)
        const uint32_t all_incl = __shfl_sync(kFull, incl, 31);
        if (!((all_incl & 0xFFFFFu) <= min(remaining, cap) && (all_incl >> 20) <= uint32_t(kIterMatches) && cur + (ca - wa) <= slen)) {
            jexec = 0;
            const uint32_t gabs = cur + myrel;
            uint32_t a = gabs + 1;
            bool stop = false;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const bool lit = ((f >> (7 - j)) & 1) == 0;
                const uint32_t n = sel(b1v[j]);
                uint32_t need, next_a;
                if (K == K_YAZ0) {
                    need = a + (lit ? 1u : 2u);   // the extended-length byte is optional (ReadByte)
                    next_a = need + ((!lit && n == 0) ? 1u : 0u);
                } else {
                    need = a + (lit ? 1u : (n == 0 ? 3u : n == 1 ? 4u : 2u));
                    next_a = need;
                }
                const bool want = orel[j] < lim;
                const bool bad = gabs >= slen || need > slen;
                if (!stop && want && bad) eos_here = true;
                stop = stop || !want || bad;
                if (!stop) jexec = j + 1;
                a = next_a;
            }
        }
        if (!taken) {
            jexec = 0;
            eos_here = false;
        }
        const uint32_t eosmask = __ballot_sync(kFull, eos_here);
        if (eosmask) {
            const uint32_t gb = __ffs(eosmask) - 1;
            if (lane > gb) jexec = 0;
            status = AURORA_END_OF_STREAM;
        }
        nlan = __popc(__ballot_sync(kFull, jexec > 0));
        break;
      }
        if (nlan == 0) {
            if (kFour && status == AURORA_OK && __shfl_sync(kFull, gsize, 0) > sink.cap()) {
                // long-group path: the first group alone exceeds the iteration budget (matches of up to 65 808 bytes):
                // its 8 tokens run one at a time, long matches as periodic 2 KiB segments with a drain in between
                const uint32_t rel0 = __shfl_sync(kFull, myrel, 0), f0 = __shfl_sync(kFull, f, 0);
                uint32_t a = rel0 + 1;   // relative to cur
                bool done = false;
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const uint32_t b1 = __shfl_sync(kFull, b1v[j], 0), l = __shfl_sync(kFull, lenv[j], 0);
                    const bool lit = ((f0 >> (7 - j)) & 1) == 0;
                    const uint32_t n = sel(b1), sz = lit ? 1u : (n == 0 ? 3u : n == 1 ? 4u : 2u);
                    if (!done && written < size) {
                        if (cur + rel0 >= slen || cur + a + sz > slen) {
                            status = AURORA_END_OF_STREAM;
                            done = true;
                        } else {
                            if (lit) {
                                sink.single_literal(written, b1);
                                written += 1;
                            } else {
                                const uint32_t ta = wa + a;
                                const uint32_t c2 = lds_u8(ta + 1), c3 = lds_u8(ta + 2), c4 = lds_u8(ta + 3);
                                uint32_t d = n == 0 ? (((c2 & 0xF) << 8) | c3) + 1 : n == 1 ? (((c3 & 0xF) << 8) | c4) + 1 : (((b1 & 0xF) << 8) | c2) + 1;
                                if (K == K_LZ40) {
                                    d = (b1 | (c2 << 8)) >> 4;
                                    if (d == 0) d = uint32_t(kWindow);   // BackCopy(0, n): one window back
                                }
                                sink.long_match(written, d, l);
                                written += l;
                            }
                            __syncwarp();
                            a += sz;
                            consumed = cur + a;
                        }
                    } else {
                        done = true;
                    }
                }
                if (status != AURORA_OK) break;
                cur += a;
                nkeep = 0;
                chain_rel = 0;
                continue;
            }
            break;
        }
        const uint32_t last = nlan - 1;
        uint32_t oend = 0, qi = qexcl, aend = 0;
        {
            uint32_t a = mya + 1;
            const uint32_t gabs1 = cur + myrel + 1;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const bool lit = ((f >> (7 - j)) & 1) == 0;
                const bool e = uint32_t(j) < jexec;
                const uint32_t b1 = b1v[j], n = sel(b1);
                const uint32_t pos = gbase + orel[j];
                uint32_t len = lenv[j], sz;
                if (K == K_YAZ0) {
                    const bool ext = !lit && n == 0;
                    const uint32_t tabs = gabs1 + (a - (mya + 1));   // blob offset of this token
                    const bool have_ext = tabs + 2 < slen;
                    if (ext && !have_ext) len = 0x11;   // Stream.ReadByte() == -1 at EOF (Yay0.cs:131)
                    sz = lit ? 1u : ((ext && have_ext) ? 3u : 2u);
                } else {
                    sz = lit ? 1u : (n == 0 ? 3u : n == 1 ? 4u : 2u);
                }
                if (e && lit) sts_u8((pos & kRingMask) | rb, b1);
                if (e && !lit) {
                    const uint32_t b2 = lds_u8(a + 1);
                    uint32_t dist = (((b1 & 0xF) << 8) | b2) + 1;
                    if (K == K_LZ11 && n == 0) dist = (((b2 & 0xF) << 8) | lds_u8(a + 2)) + 1;
                    if (K == K_LZ11 && n == 1) dist = (((lds_u8(a + 2) & 0xF) << 8) | lds_u8(a + 3)) + 1;
                    if (K == K_LZ40) {
                        dist = (b1 | (b2 << 8)) >> 4;
                        if (dist == 0) dist = uint32_t(kWindow);   // BackCopy(0, n): one window back
                    }
                    sts_u64(qaddr + 8 * qi, pos, len | (dist << 17));
                    qi++;
                }
                a += sz;
                if (e) {
                    oend = orel[j] + len;
                    aend = a - wa;
                }
            }
        }
        const uint32_t total = __shfl_sync(kFull, gexcl + oend, last);
        const uint32_t nq = __shfl_sync(kFull, qi, last);
        consumed = cur + __shfl_sync(kFull, aend, last);
        sink.submit(nq, written + total);
        written += total;
        if (status != AURORA_OK) break;
        // resume at the first group that was not executed (its start is exact: it follows exact groups)
        const uint32_t next_rel = __shfl_sync(kFull, myrel + gin, last);
        cur += next_rel;
        {   // carry the starts of the groups that did not execute
            const uint32_t carry = __shfl_down_sync(kFull, myrel, nlan & 31);
            nkeep = nvalid - nlan;
            __syncwarp();
            if (lane < nkeep) sts_u32(gaddr + 4 * lane, carry - next_rel);
            chain_rel = (ca - wa) - next_rel;
            __syncwarp();
        }
    }
    sink.finish(written);
    if (status == AURORA_OK && written > size) status = AURORA_SIZE_MISMATCH;
    return BodyResult{status, written, consumed};
}

// ---------------------------------------------------------------------------------------------
// G32 core for the split-stream formats MIO0 (MIO0.cs:105-149) and Yay0 (Yay0.cs:110-144): flags, 2-byte codes and
// literals (+ Yay0's extended-length bytes) are three sub-streams, so there is no serial chain at all: lane g takes
// flag byte g, a scan of the match counts gives its code cursor, (Yay0) a scan of its 3-byte-token count gives its
// literal cursor, and a third scan of the group output sizes gives its output base.
//   in[0] flags (relative to blob offset 0x10), in[1] codes (relative to comp_off), in[2] literals (relative to lit_off)
// ---------------------------------------------------------------------------------------------
template <int K, class Sink>
__device__ BodyResult decode_body_g32_split(InStream* in, Sink& sink, const uint32_t slen, const uint32_t size,
                                            const uint32_t comp_off, const uint32_t lit_off) {
    const uint32_t lane = lane_id();
    const uint32_t rb = sink.rbase;
    uint32_t written = 0, cur = 0, ccur = 0, lcur = 0;
    int status = AURORA_OK;

    while (written < size) {
        in[0].ensure(cur, 64);
        in[1].ensure(ccur, kInMirror - 16);
        in[2].ensure(lcur, kInMirror - 16);
        const uint32_t fa = smem_u32(in[0].window(cur)), ca = smem_u32(in[1].window(ccur)), la = smem_u32(in[2].window(lcur));
        const uint32_t f = lds_u8(fa + lane);
        const uint32_t m = f ^ 0xFFu;   // match bits, MSB first
        // ---- 256 literals in a row (random / incompressible stretches): one contiguous copy out of the literal stream
        if (__all_sync(kFull, m == 0) && size - written >= 256 && 0x10 + cur + 32 <= slen && lit_off + lcur + 256 <= slen) {
            sink.acquire_deferred(256);
            const uint32_t t = written + 8 * lane, sa = la + 8 * lane;
            if ((written & kRingMask) <= uint32_t(kRing - 256)) {
                const uint32_t ta = (t & kRingMask) | rb;
#pragma unroll
                for (int j = 0; j < 8; j++) sts_u8(ta + j, lds_u8(sa + j));
            } else {
#pragma unroll
                for (int j = 0; j < 8; j++) sts_u8(((t + j) & kRingMask) | rb, lds_u8(sa + j));
            }
            written += 256;
            cur += 32;
            lcur += 256;
            sink.submit_deferred(0, written);
            continue;
        }
        const uint32_t nm = __popc(m);
        const uint32_t mincl = warp_incl_scan(nm);
        const uint32_t mb = mincl - nm;   // matches before my group
        // my codes' first bytes (and, Yay0, how many of them are 3-byte tokens)
        uint32_t c1v[8];
        uint32_t next = 0;
        {
            uint32_t k = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const bool ism = (m >> (7 - j)) & 1;
                c1v[j] = lds_u8(ca + 2 * (mb + k));
                if (K == K_YAY0 && ism && (c1v[j] >> 4) == 0) next++;
                k += ism ? 1 : 0;
            }
        }
        uint32_t eb = 0;   // extended-length bytes before my group (they live in the literal stream)
        if (K == K_YAY0) eb = warp_incl_scan(next) - next;
        const uint32_t lb = 8 * lane - mb + eb;   // literal-stream bytes before my group
        // ---- pass 1: sizes
        uint32_t lenv[8], orel[8], litv[8];
        uint32_t gsize = 0;
        {
            uint32_t li = lb;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const bool ism = (m >> (7 - j)) & 1;
                const uint32_t n = c1v[j] >> 4;
                const bool ext = K == K_YAY0 && ism && n == 0;
                const bool extc = ext && lit_off + lcur + li < slen;   // ReadByte() == -1 at EOF: length 0x11, nothing consumed
                const uint32_t v = lds_u8(la + li);   // literal value or extended length
                litv[j] = v;
                orel[j] = gsize;
                if (K == K_MIO0) lenv[j] = ism ? n + 3 : 1;
                else lenv[j] = !ism ? 1u : (ext ? (extc ? v + 0x12u : 0x11u) : n + 2u);
                gsize += lenv[j];
                li += (!ism || ext) ? 1 : 0;   // raw count: once the literal stream is exhausted every later byte is too
            }
        }
        const uint32_t gincl = warp_incl_scan(gsize), gexcl = gincl - gsize;
        const uint32_t remaining = size - written;
        const uint32_t gbase = written + gexcl;
        const uint32_t qaddr = sink.acquire();   // the first ring / queue store of the iteration is below
        uint32_t jexec, nlan;
      for (;;) {
        const uint32_t cap = sink.cap();
        const bool taken = gexcl < remaining && gincl <= cap && mincl <= uint32_t(kIterMatches);
        const uint32_t lim = remaining - gexcl;
        // ---- which of my tokens execute
        jexec = 8;
        bool eos_here = false;
        // fast path: all 256 tokens execute (not the end of the output, all three sub-streams have their bytes)
        const uint32_t all_out = __shfl_sync(kFull, gincl, 31), all_m = __shfl_sync(kFull, mincl, 31);
        const uint32_t all_l = 256 - all_m + ((K == K_YAY0) ? __shfl_sync(kFull, eb + next, 31) : 0u);
        if (!(all_out <= min(remaining, cap) && all_m <= uint32_t(kIterMatches) && 0x10 + cur + 32 <= slen && comp_off + ccur + 2 * all_m <= slen &&
              lit_off + lcur + all_l <= slen)) {
            jexec = 0;
            const bool fbad = 0x10 + cur + lane >= slen;
            uint32_t k = 0, li = lb;
            bool stop = false;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const bool ism = (m >> (7 - j)) & 1;
                const bool ext = K == K_YAY0 && ism && (c1v[j] >> 4) == 0;
                const bool want = orel[j] < lim;
                const bool bad = fbad || (ism ? comp_off + ccur + 2 * (mb + k) + 2 > slen : lit_off + lcur + li + 1 > slen);
                if (!stop && want && bad) eos_here = true;
                stop = stop || !want || bad;
                if (!stop) jexec = j + 1;
                k += ism ? 1 : 0;
                li += (!ism || ext) ? 1 : 0;
            }
        }
        if (!taken) {
            jexec = 0;
            eos_here = false;
        }
        const uint32_t eosmask = __ballot_sync(kFull, eos_here);
        if (eosmask) {
            const uint32_t gb = __ffs(eosmask) - 1;
            if (lane > gb) jexec = 0;
            status = AURORA_END_OF_STREAM;
        }
        nlan = __popc(__ballot_sync(kFull, jexec > 0));
        break;
      }
        if (nlan == 0) break;
        const uint32_t last = nlan - 1;
        // ---- pass 2
        uint32_t oend = 0, qi = mb, kend = 0, lend = 0;
        {
            uint32_t k = 0, li = lb;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const bool ism = (m >> (7 - j)) & 1;
                const bool e = uint32_t(j) < jexec;
                const bool ext = K == K_YAY0 && ism && (c1v[j] >> 4) == 0;
                const uint32_t pos = gbase + orel[j];
                const uint32_t len = lenv[j];
                if (e && !ism) sts_u8((pos & kRingMask) | rb, litv[j]);
                if (e && ism) {
                    const uint32_t b2 = lds_u8(ca + 2 * (mb + k) + 1);
                    sts_u64(qaddr + 8 * qi, pos, len | (((((c1v[j] & 0xF) << 8) | b2) + 1) << 17));
                    qi++;
                }
                k += ism ? 1 : 0;
                li += (!ism || ext) ? 1 : 0;
                if (e) {
                    oend = orel[j] + len;
                    kend = mb + k;
                    lend = li;
                }
            }
        }
        const uint32_t total = __shfl_sync(kFull, gexcl + oend, last);
        const uint32_t nq = __shfl_sync(kFull, kend, last);
        const uint32_t nl = __shfl_sync(kFull, lend, last);
        sink.submit(nq, written + total);
        written += total;
        ccur += 2 * nq;
        {
            const uint32_t lavail = slen > lit_off + lcur ? slen - (lit_off + lcur) : 0u;
            lcur += min(nl, lavail);   // extended-length reads at EOF consumed nothing
        }
        cur += nlan;
        if (status != AURORA_OK) break;
    }
    sink.finish(written);
    if (status == AURORA_OK && written > size) status = AURORA_SIZE_MISMATCH;
    return BodyResult{status, written, max(comp_off + ccur, lit_off + lcur)};
}

// pre-history of the window: zeros (LzWindows.cs:53 rents an uncleared array; see DESIGN.md) or LZSS initialFill
__device__ __forceinline__ void ring_prefill(uint8_t* ring, uint32_t fill) {
    const uint32_t w = fill * 0x01010101u;
    const uint4 v = make_uint4(w, w, w, w);
    uint4* p = reinterpret_cast<uint4*>(ring + (kRing - kWindow));
    for (int i = lane_id(); i < kWindow / 16; i += 32) p[i] = v;
    __syncwarp();
}

template <int K, class Sink>
__device__ void decode_stream(const DecodeParams& P, uint32_t idx, InStream* in, uint8_t* ring, Sink& sink, uint32_t gaddr) {
    const uint32_t lane = lane_id();
    const uint8_t* src = P.src_base + P.src_off[idx];
    const uint64_t slen64 = P.src_len[idx];
    const uint32_t slen = slen64 > 0xFFFFFFF0ull ? 0xFFFFFFF0u : uint32_t(slen64);
    uint8_t* dst = P.dst_base + P.dst_off[idx];
    uint64_t cap = P.dst_cap[idx];
    const bool headerless = P.headerless != 0 && (K == K_LZ10 || K == K_LZ11 || K == K_LZSS);
    const uint32_t given_size = uint32_t(cap >> 32);
    if (headerless) cap &= 0xFFFFFFFFull;

    // ---- header (<= 16 bytes), read straight from global memory
    const uint32_t hb = (lane < 16 && lane < slen) ? src[lane] : 0u;
    auto H = [&](int j) { return __shfl_sync(kFull, hb, j); };
    auto be32 = [&](int j) { return (H(j) << 24) | (H(j + 1) << 16) | (H(j + 2) << 8) | H(j + 3); };
    auto le32 = [&](int j) { return H(j) | (H(j + 1) << 8) | (H(j + 2) << 16) | (H(j + 3) << 24); };

    int status = AURORA_OK;
    uint32_t size = 0, body_off = 0, comp_off = 0, lit_off = 0, consumed = 0;
    bool yaz_retry = false;

    if (headerless) {
        size = given_size;   // DecompressHeaderless(source, destination, decomLength): LZ10.cs:82, LZ11.cs:83, LZSS.cs:91
    } else if (K == K_LZ10 || K == K_LZ11 || K == K_LZ40) {
        const uint32_t id = (K == K_LZ10) ? 0x10 : (K == K_LZ11) ? 0x11 : (P.format == AURORA_FMT_LZ60 ? 0x60 : 0x40);
        if (slen < 1) { status = AURORA_END_OF_STREAM; consumed = slen; }
        else if (H(0) != id) { status = AURORA_INVALID_IDENTIFIER; consumed = 1; }
        else if (slen < 4) { status = AURORA_END_OF_STREAM; consumed = slen; }
        else {
            size = H(1) | (H(2) << 8) | (H(3) << 16);
            body_off = 4;
            if (size == 0) {
                if (slen < 8) { status = AURORA_END_OF_STREAM; consumed = slen; }
                else { size = le32(4); body_off = 8; }
            }
        }
    } else if (K == K_SMSR) {   // SMSR00.cs:49-57
        if (slen < 6) { status = AURORA_END_OF_STREAM; consumed = slen; }
        else if (H(0) != 'S' || H(1) != 'M' || H(2) != 'S' || H(3) != 'R' || H(4) != '0' || H(5) != '0') { status = AURORA_INVALID_IDENTIFIER; consumed = 6; }
        else if (slen < 16) { status = AURORA_END_OF_STREAM; consumed = slen; }
        else {
            size = be32(8);
            lit_off = be32(12);
            body_off = 16;
            if (lit_off < 16 || lit_off > 0x7FFFFFFFu) { status = AURORA_INVALID_DATA; consumed = 16; }   // ArrayPool.Rent(negative)
            else if (lit_off > slen) { status = AURORA_END_OF_STREAM; consumed = slen; }                  // ReadExactly
            else comp_off = (lit_off - 16) & ~1u;   // the ushort span: an odd trailing byte is not addressable
        }
    } else if (K == K_HUDSON) {   // LZHudson.cs:41-45: u32 big-endian size, no identifier
        if (slen < 4) { status = AURORA_END_OF_STREAM; consumed = slen; }
        else { size = be32(0); body_off = 4; }
    } else if (K == K_YAZ0 || K == K_LZSS || K == K_MIO0 || K == K_YAY0) {
        uint32_t magic;
        if (K == K_YAZ0) magic = P.format == AURORA_FMT_YAZ1 ? 0x59617A31u : 0x59617A30u;   // "Yaz1" / "Yaz0"
        else if (K == K_LZSS) magic = 0x4C5A5353u;                                           // "LZSS"
        else if (K == K_MIO0) magic = 0x4D494F30u;                                           // "MIO0"
        else magic = 0x59617930u;                                                            // "Yay0"
        if (slen < 4) { status = AURORA_END_OF_STREAM; consumed = slen; }
        else if (be32(0) != magic) { status = AURORA_INVALID_IDENTIFIER; consumed = 4; }
        else if (slen < 16) { status = AURORA_END_OF_STREAM; consumed = slen; }
        else {
            body_off = 16;
            if (K == K_LZSS) {
                size = be32(4);
            } else if (K == K_YAZ0) {
                const bool big = P.byte_order != AURORA_ENDIAN_LITTLE;   // Yaz0.cs:30 default Big
                size = big ? be32(4) : le32(4);
                yaz_retry = true;
            } else {
                bool big;
                if (P.byte_order == AURORA_ENDIAN_LITTLE) big = false;
                else if (P.byte_order == AURORA_ENDIAN_BIG) big = true;
                else {
                    // DetectByteOrder<uint>(3) stand-in: first plausible order, Big preferred (see DESIGN.md)
                    const uint32_t cb = be32(8), lb = be32(12), cl = le32(8), ll = le32(12);
                    const bool pb = cb >= 0x10 && cb <= lb && lb <= slen;
                    const bool pl = cl >= 0x10 && cl <= ll && ll <= slen;
                    big = pb || !pl;
                }
                size = big ? be32(4) : le32(4);
                comp_off = big ? be32(8) : le32(8);
                lit_off = big ? be32(12) : le32(12);
                if (K == K_YAY0 && P.byte_order == AURORA_ENDIAN_DEFAULT) (void)0;
                if (comp_off < 0x10 || comp_off > slen || lit_off < 0x10 || lit_off > slen) {
                    status = AURORA_INVALID_DATA;   // Span.Slice -> ArgumentOutOfRangeException
                    consumed = slen;
                }
            }
        }
    }

    uint32_t written = 0;
    if (status == AURORA_OK) {
        for (int attempt = 0; attempt < 2; attempt++) {
            if (uint64_t(size) > cap) {   // destination.SetLength on a non-expandable stream
                status = AURORA_DST_TOO_SMALL;
                written = 0;
                consumed = (K == K_MIO0 || K == K_YAY0) ? slen : (K == K_SMSR) ? lit_off : body_off;   // SMSR00: SetLength follows ReadExactly
            } else {
                const uint32_t fill = K == K_LZSS ? uint32_t(P.lzss.initial_fill) & 0xFFu : 0u;
                const uint32_t limit = uint32_t(min(uint64_t(0xFFFFFFFFu), cap));
                if constexpr (K == K_MIO0 || K == K_YAY0) {
                    in[0].begin(P.src_base, P.src_limit, src + 0x10);
                    in[1].begin(P.src_base, P.src_limit, src + comp_off);
                    in[2].begin(P.src_base, P.src_limit, src + lit_off);
                } else if constexpr (K == K_SMSR) {
                    in[0].begin(P.src_base, P.src_limit, src + 0x10);
                    in[1].begin(P.src_base, P.src_limit, src + lit_off);
                } else {
                    in[0].begin(P.src_base, P.src_limit, src);
                }
                BodyResult r;
                bool g32 = K != K_HUDSON && K != K_SMSR;
                if (K == K_LZSS) g32 = 8u * (((1u << P.lzss.length_bits) - 1u) + uint32_t(P.lzss.min_length)) <= uint32_t(kSubMaxG);
                if (g32) {
                    if constexpr (K != K_HUDSON && K != K_SMSR) {
                    sink.begin(ring, fill, dst, limit);
                    if constexpr (K == K_MIO0 || K == K_YAY0) r = decode_body_g32_split<K>(in, sink, slen, size, comp_off, lit_off);
                    else if constexpr (K == K_YAZ0 || K == K_LZ11 || K == K_LZ40) r = decode_body_g32_var<K>(in, sink, gaddr, slen, size, body_off);
                    else r = decode_body_g32<K>(in, sink, gaddr, slen, size, body_off, P.lzss);
                    }
                } else if constexpr (K == K_LZSS || K == K_HUDSON || K == K_SMSR) {
                    // LzProperties whose largest group exceeds an iteration, LZHudson (a 32-bit flag word is exactly one
                    // 32-token iteration) and SMSR00: the token-per-lane core, run by this warp alone
                    sink.wait_idle();
                    ring_prefill(ring, fill);
                    OutState out;
                    out.ring = ring;
                    out.rbase = smem_u32(ring);
                    out.dst = dst;
                    out.limit = limit;
                    out.flushed = 0;
                    out.aligned = (reinterpret_cast<uintptr_t>(dst) & 15) == 0;
                    r = decode_body<K>(in, out, slen, size, body_off, comp_off, lit_off, P.lzss);
                }
                status = r.status;
                written = r.written;
                consumed = r.consumed;
                if (status == AURORA_END_OF_STREAM) consumed = slen;
                if ((K == K_MIO0 || K == K_YAY0) && status != AURORA_OK) consumed = slen;
            }
            // Yaz0.cs:67-78: on any exception retry once with the byte-swapped size
            if (!(yaz_retry && attempt == 0 && status != AURORA_OK)) break;
            size = bswap32(size);
            status = AURORA_OK;
        }
    }
    if (lane == 0) {
        P.out_len[idx] = written;
        P.consumed[idx] = consumed;
        P.status[idx] = status;
    }
}

// ---- kernel
template <int K>
__global__ void __launch_bounds__(Traits<K>::kSlots * 64, Traits<K>::kBlocksPerSM) decode_flaglz_kernel(const DecodeParams P) {
    using T = Traits<K>;
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5;
#ifdef AURORA_AFFINE
    // developer probe: roles by scheduler (warps 4k, 4k+1 parse, 4k+2, 4k+3 resolve; a warp runs on scheduler warp % 4), no register split
    const int role = (warp >> 1) & 1;
    const int slot = (warp >> 2) * 2 + (warp & 1);
#else
    // warpgroups alternate parser / resolver; slot s is served by parser warp (s / 4) * 8 + s % 4 and the warp 4 above it
    const int role = (warp >> 2) & 1;
    const int slot = (warp >> 3) * 4 + (warp & 3);
#endif
    // rings first, 8 KiB aligned in the shared window (wrapped ring addresses become one LOP3); the launcher adds 8 KiB of slack
    const uint32_t s0 = smem_u32(smem);
    uint8_t* aligned = smem + (((s0 + kRing - 1) & ~uint32_t(kRing - 1)) - s0);
    uint8_t* ring = aligned + size_t(slot) * kRing;
    uint8_t* aux = aligned + size_t(T::kSlots) * kRing + size_t(slot) * T::kAuxBytes;
    uint8_t* qptr = aux + T::kStreams * kInStage;
    const uint32_t qbase = smem_u32(qptr), gaddr = qbase + T::kQueueBytes, mail = gaddr + 128;
    uint64_t* bars = reinterpret_cast<uint64_t*>(qptr + T::kQueueBytes + 128 + 48);
    const uint32_t bar_f = 2 * slot, bar_e = 2 * slot + 1;   // the slot's two named barriers (no __syncthreads in this kernel)

    if (role == 0) {
        if constexpr (T::kRegSplit) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(T::kParserRegs));
        InStream in[T::kStreams];
#pragma unroll
        for (int s = 0; s < T::kStreams; s++) in[s].init(aux + s * kInStage, bars + 2 * s);
        fence_proxy_async();
        __syncwarp();   // the slot's TMA mbarriers are initialised (only this warp uses them)
        SlotSink sink;
        sink.rbase = smem_u32(ring);
        sink.qbase = qbase;
        sink.mail = mail;
        sink.bar_f = bar_f;
        sink.bar_e = bar_e;
        sink.init();
        for (;;) {
            uint32_t t = 0;
            if (lane_id() == 0) t = atomicAdd(P.ticket, 1u);
            t = __shfl_sync(kFull, t, 0);
            if (t >= P.n) break;
            const uint32_t idx = P.order ? P.order[t] : t;
            decode_stream<K>(P, idx, in, ring, sink, gaddr);
        }
        sink.exit();
#pragma unroll
        for (int s = 0; s < T::kStreams; s++) in[s].drain_inflight();
    } else {
        if constexpr (T::kRegSplit) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(T::kResolverRegs));
        resolver_role(ring, qbase, mail, bar_f, bar_e);
    }
}

template <int K>
cudaError_t launch(const DecodeParams& p, int sm_count, cudaStream_t st) {
    using T = Traits<K>;
    static_assert(T::kSlots == 4 || T::kSlots == 8, "a block has 16 named barriers: at most 8 slots, in warpgroups of 4");
    const int threads = T::kSlots * 64;
    const size_t smem = size_t(T::kSmemPerBlock);
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!configured[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(decode_flaglz_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
        if (e != cudaSuccess) return e;
        configured[dev & 63] = true;
    }
    int blocks = sm_count * T::kBlocksPerSM;
    const int needed_blocks = int((p.n + T::kSlots - 1) / T::kSlots);
    if (needed_blocks < blocks) blocks = needed_blocks > 0 ? needed_blocks : 1;
    decode_flaglz_kernel<K><<<blocks, threads, smem, st>>>(p);
    return cudaGetLastError();
}

}  // namespace

cudaError_t launch_decode_flaglz(const DecodeParams& p, int sm_count, cudaStream_t st) {
    switch (p.format) {
        case AURORA_FMT_LZ10: return launch<K_LZ10>(p, sm_count, st);
        case AURORA_FMT_LZ11: return launch<K_LZ11>(p, sm_count, st);
        case AURORA_FMT_YAZ0:
        case AURORA_FMT_YAZ1: return launch<K_YAZ0>(p, sm_count, st);
        case AURORA_FMT_LZSS: return launch<K_LZSS>(p, sm_count, st);
        case AURORA_FMT_MIO0: return launch<K_MIO0>(p, sm_count, st);
        case AURORA_FMT_YAY0: return launch<K_YAY0>(p, sm_count, st);
        case AURORA_FMT_LZHUDSON: return launch<K_HUDSON>(p, sm_count, st);
        case AURORA_FMT_LZ40:
        case AURORA_FMT_LZ60: return launch<K_LZ40>(p, sm_count, st);
        case AURORA_FMT_SMSR00: return launch<K_SMSR>(p, sm_count, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace aurora
