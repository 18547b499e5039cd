// encode_lz_par.cu — the window match search of the flag-byte encoders with ONE LANE PER WINDOW POSITION and shared-memory
// hash tables (LZ10 / BLZ, LZ11 / LZ40 / LZ60, Yaz0 / Yaz1, LZSS, MIO0, Yay0, LZHudson, SMSR00; every quality).  One raw buffer per warp, 32 positions per step.
//
// The output is byte-identical to the reference encoder (and to the sequential replay in encode_lz.cu / finder.cuh, which
// stays for the other formats and qualities): what LzChainMatchFinder computes at a position depends only on the bytes
// before it, not on the parse —
//   * every position up to length - 4 is inserted into the head / chain tables, in order, whether it is searched
//     (MatchSearch, LzChainMatchFinder.cs:214-246) or lies inside a match (the insert loop of FindNextBestMatch, :196-205);
//   * so the candidates of position p are exactly the earlier positions with the same hash value, nearest first, at most
//     maxChain of them, until the distance exceeds MaxDistance (ChainMatches, :248-282) — a function of the data alone.
// The search can therefore run at ALL positions in parallel, and the reference's greedy parse with its one-step lazy
// lookahead (:157-212) becomes a cheap walk over the per-position results.
//
// Tables (20 KiB of shared memory per warp instead of the reference's 2 MiB head table per stream):
//   data[8192]  u8   ring of the raw bytes (window + step + lookahead), refilled 512 bytes at a time with 16-byte loads;
//   head[2048]  u16  latest position (mod 2^16) whose hash falls into the bucket = low 11 bits of the reference's hash;
//   node[4096]  u16  ring over the last 4096 positions: distance to the previous position of the same BUCKET (0: none) in
//                    13 bits and three of the reference's remaining hash bits above — a chain node counts as a candidate
//                    (and as one of the maxChain attempts) only when its whole hash value equals the searching position's
//                    (the three bits reject most foreign nodes, the rest are confirmed by hashing the node's four bytes
//                    again), which reproduces the reference's per-hash-value chains exactly.
// Positions of the step that is being searched are not in the ring yet (they would overwrite the far end of the window):
// the candidates among them are the lanes with the same hash value (match.any), walked as a bit mask.
// Per step: hashes, bucket groups (match.any), chain walk with a word-wise common-prefix comparison per candidate, ring
// update; the parse of the PREVIOUS step (its lazy test needs the first result of this one) walks only the matches —
// literal runs are mask operations — and all tokens of a step are written at once: one warp scan gives byte offsets, flag
// bytes are assembled with match.any / redux.or per group of eight tokens.
#include "common.cuh"
#include "stage.cuh"

namespace aurora {

namespace {

#ifndef AURORA_ENC_BUCKET_BITS
#define AURORA_ENC_BUCKET_BITS 11
#endif
#ifndef AURORA_ENC_DATA
#define AURORA_ENC_DATA 5120
#endif
constexpr int kBucketBits = AURORA_ENC_BUCKET_BITS, kBuckets = 1 << kBucketBits, kBucketMask = kBuckets - 1;
constexpr int kWin = 4096, kWinMask = kWin - 1;
// ring of the raw bytes: the 4 KiB window, the step, the longest lookahead (max_length <= 288) and the refill granularity
// (512 + 16 bytes) need 4936 bytes; the index is a modulo by a constant (a multiply-high), not a mask: 5 KiB instead of 8 KiB
// per warp is two more resident warps per SM, and the kernel is latency bound (measured at quality 8, LZ10 / Yaz0 GB/s raw in: 8 KiB ring
// + 2048 buckets = 11 warps 12.5 / 13.5; 5 KiB + 2048 = 13 warps 13.3 / 14.0; 5 KiB + 1024 buckets = 15 warps 12.4 / 12.7)
constexpr uint32_t kData = AURORA_ENC_DATA;
__device__ __forceinline__ uint32_t didx(uint32_t x) { return x % kData; }
constexpr int kLook = 288;                // bytes behind a position the ring guarantees (the longest match of every format but the LZ11 family)
constexpr int kChunk = 512;              // raw bytes staged per refill (16 bytes per lane)
// head + node ring + data; qualities >= 10 add a second head / node ring pair for the reference's small-match table
// (`M`: LzChainMatchFinder.cs:85-91, :236-244 — the latest position whose first min_length bytes hash to the same 16-bit value)
template <bool M>
constexpr int kTablesPerWarp = (kBuckets * 2 + kWin * 2) * (M ? 2 : 1) + int(kData);
template <bool M>
constexpr int kParWarps = (227 * 1024) / kTablesPerWarp<M> > 16 ? 16 : (227 * 1024) / kTablesPerWarp<M>;   // one block per SM

enum ParKind { P_LZ10 = 0, P_YAZ0 = 1, P_LZSS = 2, P_MIO0 = 3, P_YAY0 = 4, P_LZ11 = 5, P_HUDSON = 6, P_SMSR = 7 };   // P_LZ11: LZ11 / LZ40 / LZ60
// tokens per flag word: LZHudson writes Yaz0's tokens under 32-bit big-endian flag words (LZHudson.cs:48-59), SMSR00 MIO0's
// codes under 16-bit ones with the literals in a section of their own (SMSR00.cs:60-75); everything else has flag bytes
template <int K>
constexpr uint32_t kGroup = K == P_HUDSON ? 32u : K == P_SMSR ? 16u : 8u;
// MIO0 / Yay0 write three sections (flag bytes, match codes, literal bytes: MIO0.cs:159-184, Yay0.cs:152-184)
template <int K>
constexpr bool kSplit = K == P_MIO0 || K == P_YAY0;

struct ParState {
    // tables (shared addresses)
    uint32_t head, node, data;
    uint32_t head2, node2;   // small-match table (qualities >= 10): buckets and chains over the 16-bit hash of the first min_length bytes
    uint32_t min_mask;
    uint32_t skew;           // ring index of position 0 (the source's offset inside its 16-byte line)
    int staged;              // positions below this are in the data ring
    // source
    const uint8_t* src;
    const uint8_t* src_lim;        // 16-byte lines starting below this may be read
    int n, limit;
    // finder parameters
    int hash_shift, max_chain, lazy, min_len, max_len, min_dist, max_dist;
    uint32_t hash_mask;
    int look;                // min(max_len, kLook): prefix comparisons inside the data ring; longer ones continue in global memory
    bool no_self_overlap, blz, lz40;
    // output
    uint8_t* out;
    uint64_t cap, pos;
    uint32_t ntok;         // tokens written so far
    uint32_t carry_flag;   // bits of the open flag group
    uint64_t carry_pos;    // ... and where its byte lives
    bool overflow;
    // parse state: offset of the next token start relative to the step that is parsed next, and whether that token is the
    // match the lazy test already chose
    int cur_off;
    bool forced, pending;
    // LZSS token fields
    int lz_n, lz_f, lz_start, lz_lbits;
    // MIO0 / Yay0: the code and literal sections are staged in this warp's slice of the global scratch buffer until the
    // length of the flag section in front of them is known
    uint8_t* scratch;
    uint8_t* codes;
    uint8_t* lits;
    uint32_t ncodes, nlits;
    uint64_t flag_base;    // first byte of the flag section (one byte per eight tokens)
};

__device__ __forceinline__ uint32_t ring_u8(const ParState& S, int pos) { return lds_u8(S.data + didx(uint32_t(pos) + S.skew)); }

// the ring index 4 bytes further (indices are multiples of 4 here, the ring size is too: no straddling)
__device__ __forceinline__ uint32_t dnext(uint32_t i) {
    i += 4;
    return i >= kData ? i - kData : i;
}

// i < 2 * kData folded back into the ring
__device__ __forceinline__ uint32_t dwrap(uint32_t i) { return i >= kData ? i - kData : i; }

// four bytes at ring index i (any alignment; (i & 3) is the byte position inside the aligned word)
__device__ __forceinline__ uint32_t ring_u32_at(const ParState& S, uint32_t i) {
    const uint32_t i0 = i & ~3u;
    const uint32_t lo = lds_u32(S.data + i0), hi = lds_u32(S.data + dnext(i0));
    return __funnelshift_r(lo, hi, (i & 3u) * 8);
}
// four bytes at an arbitrary position (little-endian) from the data ring
__device__ __forceinline__ uint32_t ring_u32(const ParState& S, int pos) { return ring_u32_at(S, didx(uint32_t(pos) + S.skew)); }

// stage raw bytes until position `upto` (exclusive, clamped to the stream) is in the ring: whole 16-byte lines, 512 bytes per pass
__device__ __forceinline__ void stage(ParState& S, int upto) {
    upto = min(upto, S.n);
    while (S.staged < upto) {
        // line index l covers positions [16 l - skew, 16 l - skew + 16)
        const uint32_t first_line = (uint32_t(S.staged) + S.skew) >> 4;
        const uint32_t line = first_line + lane_id();
        const uint8_t* g = S.src - S.skew + size_t(line) * 16;
        if (g < S.src_lim) {
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(g));
            sts_u128(S.data + didx(line * 16), v.x, v.y, v.z, v.w);
        }
        S.staged = int((first_line + 32) * 16 - S.skew);
    }
    __syncwarp();
}

// common prefix of the bytes at positions a and b, at most cap bytes, the first `known` of them known to be equal
// (GetMatchLength, LzChainMatchFinder.cs:338-357)
// ia / ib: ring indices of the two strings' first bytes (one modulo per position and step; everything below is index arithmetic)
__device__ __forceinline__ int prefix_len(const ParState& S, uint32_t ia0, uint32_t ib0, int cap, int known) {
    int len = known & ~3;
    const uint32_t pa = dwrap(ia0 + uint32_t(len)), pb = dwrap(ib0 + uint32_t(len));   // (len <= max_length <= 288 < kData)
    uint32_t ia = pa & ~3u, ib = pb & ~3u;
    if (((pa ^ pb) & 3u) == 0) {
        // distance a multiple of 4 (tile data): the two byte strings have the same alignment, aligned words compare directly
        const uint32_t r = pa & 3u;
        uint32_t mask = 0xFFFFFFFFu << (8 * r);
        int l = len - int(r);
        while (l < cap) {
            const uint32_t x = (lds_u32(S.data + ia) ^ lds_u32(S.data + ib)) & mask;
            if (x) return min(l + ((__ffs(int(x)) - 1) >> 3), cap);
            mask = 0xFFFFFFFFu;
            l += 4;
            ia = dnext(ia);
            ib = dnext(ib);
        }
        return cap;
    }
    const uint32_t sha = (pa & 3u) * 8, shb = (pb & 3u) * 8;
    uint32_t wa = lds_u32(S.data + ia), wb = lds_u32(S.data + ib);
    while (len + 4 <= cap) {
        ia = dnext(ia);
        ib = dnext(ib);
        const uint32_t na = lds_u32(S.data + ia), nb = lds_u32(S.data + ib);
        const uint32_t x = __funnelshift_r(wa, na, sha) ^ __funnelshift_r(wb, nb, shb);
        if (x) return len + ((__ffs(int(x)) - 1) >> 3);
        wa = na;
        wb = nb;
        len += 4;
    }
    while (len < cap && lds_u8(S.data + dwrap(ia0 + uint32_t(len))) == lds_u8(S.data + dwrap(ib0 + uint32_t(len)))) len++;
    return len;
}

template <int K>
__device__ __forceinline__ uint32_t token_size(const ParState& S, int len) {
    if (K == P_YAZ0 || K == P_HUDSON) return len < 18 ? 2u : 3u;
    if (K == P_LZ11) return S.lz40 ? (len < 16 ? 2u : len < 272 ? 3u : 4u) : (len <= 16 ? 2u : len <= 272 ? 3u : 4u);   // LZ40.cs:126-168, LZ11.cs:135-171
    return 2u;
}

// the common prefix beyond the ring's lookahead (LZ11 family: matches of up to 0x4000 bytes), byte by byte from the source
__device__ __noinline__ int extend_global(const uint8_t* a, int distance, int l, int cap) {
    const uint8_t* b = a - distance;
    while (l + 4 <= cap) {
        const uint32_t a0 = __ldg(a + l), a1 = __ldg(a + l + 1), a2 = __ldg(a + l + 2), a3 = __ldg(a + l + 3);
        const uint32_t b0 = __ldg(b + l), b1 = __ldg(b + l + 1), b2 = __ldg(b + l + 2), b3 = __ldg(b + l + 3);
        if (a0 != b0) return l;
        if (a1 != b1) return l + 1;
        if (a2 != b2) return l + 2;
        if (a3 != b3) return l + 3;
        l += 4;
    }
    while (l < cap && __ldg(a + l) == __ldg(b + l)) l++;
    return l;
}

// ---- the parse of one step (FindNextBestMatch, :157-212).  `len`: the search results of the step's 32 positions (0 where
// nothing was found, the position lies behind `limit`, or it was not searched because an earlier match covers it).
// Returns the literal and match token masks.  A token that starts at lane 31 with a short match needs the result of the next
// step's first position for the lazy test: it is left pending (S.pending) and resolved by the caller after the next search.
__device__ __forceinline__ void parse_step(ParState& S, int base, int len, uint32_t& lit_out, uint32_t& mat_out) {
    const uint32_t mmask = __ballot_sync(kFull, len >= S.min_len);
    uint32_t lit = 0, mat = 0;
    int c = S.cur_off;
    bool forced = S.forced;
    while (c < 32) {
        int k;
        if (forced) {
            k = c;
        } else {
            const uint32_t rest = mmask >> c;
            if (rest == 0) {
                lit |= ~0u << c;
                c = 32;
                break;
            }
            k = c + __ffs(int(rest)) - 1;
            lit |= ((1u << k) - 1u) & (~0u << c);
        }
        const int lk = __shfl_sync(kFull, len, k);
        if (!forced && lk <= S.lazy && base + k + 1 <= S.limit) {
            if (k == 31) {   // the lazy test needs the next step
                S.pending = true;
                c = 32;
                break;
            }
            const int ln = __shfl_sync(kFull, len, k + 1);
            if (ln > lk) {   // the next position has the longer match: literal here
                lit |= 1u << k;
                forced = true;
                c = k + 1;
                continue;
            }
        }
        mat |= 1u << k;
        forced = false;
        c = k + lk;
    }
    S.cur_off = c - 32;
    S.forced = forced;
    lit_out = lit;
    mat_out = mat;
}

// ---- the tokens of one step: `lit` / `mat` = the lanes that start a literal / a match token (len, dist: their results)
template <int K>
__device__ __forceinline__ void write_step(ParState& S, int base, int len, int dist, uint32_t lit, uint32_t mat) {
    const int lane = lane_id();
    const uint32_t lt = (1u << lane) - 1u;
    // positions at or behind the end of the data are no tokens
    const uint32_t inb = base + 32 <= S.n ? ~0u : (S.n > base ? (1u << (S.n - base)) - 1u : 0u);
    lit &= inb;
    mat &= inb;
    const uint32_t tok = lit | mat;
    if (tok == 0) return;
    const bool is_tok = (tok >> lane) & 1u, is_mat = (mat >> lane) & 1u;
    // ---- byte offsets: token bytes + one flag word (G / 8 bytes) in front of every G-th token
    constexpr uint32_t G = kGroup<K>, FB = G / 8;
    const uint32_t T = S.ntok + __popc(tok & lt);
    const bool opens = is_tok && (T & (G - 1u)) == 0;
    const uint32_t sz = !is_tok ? 0u : (is_mat ? token_size<K>(S, len) : (K == P_SMSR ? 0u : 1u)) + (opens ? FB : 0u);
    const uint32_t incl = warp_incl_scan(sz);
    const uint64_t at = S.pos + (incl - sz);          // first byte of my token (its flag word, when it opens a group)
    const uint64_t tb = at + (opens ? FB : 0u);       // token bytes
    const uint32_t total = __shfl_sync(kFull, incl, 31);
    // ---- flag words.  LZ10 / LZ11: 1 = match, MSB first; Yaz0 / LZHudson / SMSR00: 1 = literal, MSB first; LZSS: 1 = literal, LSB first
    {
        const bool bitv = (K == P_LZ10 || K == P_LZ11) ? is_mat : !is_mat;
        const uint32_t sh = (K == P_LZSS) ? (T & 7u) : G - 1u - (T & (G - 1u));
        const uint32_t contrib = (is_tok && bitv) ? 1u << sh : 0u;
        const uint32_t g = T / G;
        const uint32_t gm = __match_any_sync(kFull, is_tok ? g : 0xFFFFFFFFu);
        uint32_t fv = __reduce_or_sync(gm, contrib);
        const bool leader = is_tok && (gm & lt) == 0;   // first token of the group within this step
        uint64_t fpos = at;                             // a group opened in this step: the word in front of its first token
        if (leader && !opens) {                         // the group was opened by an earlier step
            fv |= S.carry_flag;
            fpos = S.carry_pos;
        }
        if (leader) {
            if (fpos + FB <= S.cap) {
                if (FB == 1) {
                    S.out[fpos] = uint8_t((K == P_LZ11 && S.lz40) ? 0u - fv : fv);   // LZ40.cs:137: (byte)-flag
                } else {
                    for (uint32_t i = 0; i < FB; i++) S.out[fpos + i] = uint8_t(fv >> (8 * (FB - 1 - i)));   // big-endian word
                }
            } else {
                for (uint32_t i = 0; i < FB; i++)
                    if (fpos + i < S.cap) S.out[fpos + i] = uint8_t(fv >> (8 * (FB - 1 - i)));
                S.overflow = true;
            }
        }
        // carry the last group when it is still open
        const uint32_t ntok = __popc(tok);
        const int last = 31 - __clz(int(tok));
        const uint32_t lead_lane = __ffs(int(__shfl_sync(kFull, gm, last))) - 1;
        const uint32_t cf = __shfl_sync(kFull, fv, lead_lane);
        const uint32_t cplo = __shfl_sync(kFull, uint32_t(fpos), lead_lane), cphi = __shfl_sync(kFull, uint32_t(fpos >> 32), lead_lane);
        S.ntok += ntok;
        S.carry_flag = (S.ntok & (G - 1u)) ? cf : 0u;
        S.carry_pos = uint64_t(cplo) | (uint64_t(cphi) << 32);
    }
    // ---- token bytes
    if (is_tok) {
        uint32_t b0, b1, b2 = 0, b3 = 0, nb;
        if (!is_mat) {
            b0 = ring_u8(S, base + lane);
            b1 = 0;
            nb = 1;
            if (K == P_SMSR) {   // the literal section, in token order
                S.lits[S.nlits + __popc(lit & lt)] = uint8_t(b0);
                nb = 0;
            }
        } else if (K == P_SMSR) {
            const uint32_t v = (uint32_t(dist - 1) | uint32_t(len - 3) << 12) & 0xFFFFu;   // MIO0's code
            b0 = v >> 8;
            b1 = v & 0xFF;
            nb = 2;
        } else if (K == P_LZ10) {
            const uint32_t v = uint32_t(len - 3) << 12 | (uint32_t(dist - (S.blz ? 3 : 1)) & 0xFFFu);   // BLZ.cs: distance - 3
            b0 = (v >> 8) & 0xFF;
            b1 = v & 0xFF;
            nb = 2;
        } else if (K == P_LZ11 && S.lz40) {
            // (ushort)(Distance << 4 | ...), little-endian: a distance of 0x1000 truncates to 0
            const uint32_t dd = (uint32_t(dist) << 4) & 0xFFFFu;
            b1 = dd >> 8;
            if (len < 16) {
                b0 = (dd | uint32_t(len)) & 0xFF;
                nb = 2;
            } else if (len < 272) {
                b0 = dd & 0xFF;
                b2 = uint32_t(len - 16) & 0xFF;
                nb = 3;
            } else {
                b0 = (dd | 1u) & 0xFF;
                b2 = uint32_t(len - 272) & 0xFF;
                b3 = (uint32_t(len - 272) >> 8) & 0xFF;
                nb = 4;
            }
        } else if (K == P_LZ11) {
            const uint32_t d1 = uint32_t(dist - 1) & 0xFFFu;
            if (len <= 16) {
                const uint32_t v = (uint32_t(len - 1) << 12 | d1) & 0xFFFFu;
                b0 = v >> 8;
                b1 = v & 0xFF;
                nb = 2;
            } else if (len <= 272) {
                const uint32_t v = (uint32_t(len - 17) << 12 | d1) & 0xFFFFu;
                b0 = (uint32_t(len - 17) & 0xFF) >> 4;
                b1 = v >> 8;
                b2 = v & 0xFF;
                nb = 3;
            } else {
                const uint32_t v = 0x10000000u | (uint32_t(len - 273) & 0xFFFFu) << 12 | d1;
                b0 = v >> 24;
                b1 = (v >> 16) & 0xFF;
                b2 = (v >> 8) & 0xFF;
                b3 = v & 0xFF;
                nb = 4;
            }
        } else if (K == P_YAZ0 || K == P_HUDSON) {
            const uint32_t d1 = uint32_t(dist - 1) & 0xFFFu;
            if (len < 18) {
                const uint32_t v = (uint32_t(dist - 1) | uint32_t(len - 2) << 12) & 0xFFFFu;
                b0 = v >> 8;
                b1 = v & 0xFF;
                nb = 2;
            } else {
                b0 = d1 >> 8;
                b1 = d1 & 0xFF;
                b2 = uint32_t(len - 0x12) & 0xFF;
                nb = 3;
            }
        } else {
            // LZSS.cs:132-160: the token holds the ring offset of the source, sp = position behind... of the match start
            const int offset = (S.lz_start + (base + lane) - dist) & S.lz_n;
            const uint32_t v = (uint32_t(offset & 0xFF) | uint32_t(offset & 0xFF00) << S.lz_lbits | uint32_t((len - S.min_len) & S.lz_f) << 8) & 0xFFFFu;
            b0 = v & 0xFF;
            b1 = v >> 8;
            nb = 2;
        }
        if (tb + nb <= S.cap) {
            if (nb > 0) S.out[tb] = uint8_t(b0);
            if (nb > 1) S.out[tb + 1] = uint8_t(b1);
            if (nb > 2) S.out[tb + 2] = uint8_t(b2);
            if (nb > 3) S.out[tb + 3] = uint8_t(b3);
        } else {
            S.overflow = true;
        }
    }
    if (K == P_SMSR) S.nlits += __popc(lit);
    S.pos += total;
}

// ---- the same for the split formats: one flag bit per token into the flag section (1 = literal, MSB first), two code
// bytes per match into the code section; literal bytes and (Yay0, length >= 18) the extended length byte into the
// literal section, all in token order
template <int K>
__device__ __forceinline__ void write_step_split(ParState& S, int base, int len, int dist, uint32_t lit, uint32_t mat) {
    const int lane = lane_id();
    const uint32_t lt = (1u << lane) - 1u;
    const uint32_t inb = base + 32 <= S.n ? ~0u : (S.n > base ? (1u << (S.n - base)) - 1u : 0u);
    lit &= inb;
    mat &= inb;
    const uint32_t tok = lit | mat;
    if (tok == 0) return;
    const bool is_tok = (tok >> lane) & 1u, is_mat = (mat >> lane) & 1u;
    const uint32_t T = S.ntok + __popc(tok & lt);
    // ---- section offsets: literal bytes in the low half, code bytes in the high half of one scan (<= 32 / <= 64 per step)
    const bool ext = K == P_YAY0 && is_mat && len >= 18;
    const uint32_t sz = !is_tok ? 0u : is_mat ? (0x20000u | (ext ? 1u : 0u)) : 1u;
    const uint32_t incl = warp_incl_scan(sz);
    const uint32_t excl = incl - sz;
    const uint32_t total = __shfl_sync(kFull, incl, 31);
    const uint32_t lit_at = S.nlits + (excl & 0xFFFFu), code_at = S.ncodes + (excl >> 16);
    // ---- flag bytes
    {
        const uint32_t contrib = (is_tok && !is_mat) ? 0x80u >> (T & 7u) : 0u;
        const uint32_t g = T >> 3;
        const uint32_t gm = __match_any_sync(kFull, is_tok ? g : 0xFFFFFFFFu);
        uint32_t fv = __reduce_or_sync(gm, contrib);
        const bool leader = is_tok && (gm & lt) == 0;
        if (leader && (T & 7u) != 0) fv |= S.carry_flag;   // the group was opened by an earlier step
        if (leader) {
            const uint64_t fpos = S.flag_base + g;
            if (fpos < S.cap) S.out[fpos] = uint8_t(fv);
            else S.overflow = true;
        }
        const int last = 31 - __clz(int(tok));
        const uint32_t lead_lane = __ffs(int(__shfl_sync(kFull, gm, last))) - 1;
        const uint32_t cf = __shfl_sync(kFull, fv, lead_lane);
        S.ntok += __popc(tok);
        S.carry_flag = (S.ntok & 7u) ? cf : 0u;
    }
    // ---- section bytes
    if (is_tok) {
        if (!is_mat) {
            S.lits[lit_at] = uint8_t(ring_u8(S, base + lane));
        } else {
            uint32_t v;
            if (K == P_MIO0) v = (uint32_t(dist - 1) | uint32_t(len - 3) << 12) & 0xFFFFu;
            else if (len < 18) v = (uint32_t(dist - 1) | uint32_t(len - 2) << 12) & 0xFFFFu;
            else v = uint32_t(dist - 1) & 0xFFFu;
            S.codes[code_at] = uint8_t(v >> 8);
            S.codes[code_at + 1] = uint8_t(v & 0xFF);
            if (ext) S.lits[lit_at] = uint8_t(len - 0x12);
        }
    }
    S.nlits += total & 0xFFFFu;
    S.ncodes += total >> 16;
}

template <int K>
__device__ __forceinline__ void emit_step(ParState& S, int base, int len, int dist, uint32_t lit, uint32_t mat) {
    if constexpr (kSplit<K>) write_step_split<K>(S, base, len, dist, lit, mat);
    else write_step<K>(S, base, len, dist, lit, mat);
}

__device__ __forceinline__ void put_byte(ParState& S, uint32_t b) {
    if (S.pos < S.cap) {
        if (lane_id() == 0) S.out[S.pos] = uint8_t(b);
    } else {
        S.overflow = true;
    }
    S.pos++;
}
__device__ __forceinline__ void put_u32p(ParState& S, uint32_t v, bool big) {
    for (int i = 0; i < 4; i++) put_byte(S, big ? (v >> (24 - 8 * i)) & 0xFF : (v >> (8 * i)) & 0xFF);
}

template <int K, bool M>
__device__ void encode_stream_par(const EncodeParams& P, uint32_t idx, ParState& S) {
    const int lane = lane_id();
    const uint64_t n64 = P.src_len[idx];
    int status = AURORA_OK;
    uint64_t out_len = 0;
    if (n64 > 0x7FFFFFF0ull) {
        status = AURORA_INVALID_ARGUMENT;
    } else {
        const int n = int(n64);
        S.src = P.src_base + P.src_off[idx];
        S.skew = uint32_t(reinterpret_cast<uintptr_t>(S.src) & 15);
        S.src_lim = P.src_base + P.src_limit;   // (a 16-byte line that starts inside the batch's source bytes is readable)
        S.staged = 0;
        S.n = n;
        S.limit = n - 4;
        S.out = P.dst_base + P.dst_off[idx];
        S.cap = P.dst_cap[idx];
        S.pos = 0;
        S.ntok = 0;
        S.carry_flag = 0;
        S.carry_pos = 0;
        S.overflow = false;
        S.cur_off = 0;
        S.forced = false;
        S.pending = false;
        const bool big = P.byte_order != AURORA_ENDIAN_LITTLE;
        // ---- headers (as encode_lz.cu: LZ10.cs:67-80, Yaz0.cs:82-98, LZSS.cs:72-89; BLZ has none)
        if (K == P_LZ10 || K == P_LZ11) {
            if (P.format != AURORA_FMT_BLZ) {
                const uint32_t id = K == P_LZ10 ? 0x10u : P.format == AURORA_FMT_LZ40 ? 0x40u : P.format == AURORA_FMT_LZ60 ? 0x60u : 0x11u;
                if (n <= 0xFFFFFF) {
                    put_u32p(S, id | (uint32_t(n) << 8), false);
                } else {
                    put_u32p(S, id, false);
                    put_u32p(S, uint32_t(n), false);
                }
            }
        } else if (K == P_HUDSON) {
            put_u32p(S, uint32_t(n), true);   // LZHudson.cs:48-59: the size, then Yay0.CompressHeaderless under 4-byte flag words
        } else if (K == P_SMSR) {
            // SMSR00.cs:60-75: "SMSR00", u16 0, BE size, BE pointer to the literal section (patched below)
            const char* magic = "SMSR00";
            for (int i = 0; i < 6; i++) put_byte(S, uint8_t(magic[i]));
            put_byte(S, 0);
            put_byte(S, 0);
            put_u32p(S, uint32_t(n), true);
            put_u32p(S, 0, true);
            S.codes = S.scratch + P.scratch_per_warp - 2 * (size_t(n) + 64);   // (the layout of encode_lz.cu; only the literal half is used)
            S.lits = S.codes + size_t(n) + 32;
            S.ncodes = S.nlits = 0;
        } else if (K == P_YAZ0) {
            const char* magic = P.format == AURORA_FMT_YAZ1 ? "Yaz1" : "Yaz0";
            for (int i = 0; i < 4; i++) put_byte(S, uint8_t(magic[i]));
            put_u32p(S, uint32_t(n), big);
            put_u32p(S, P.yaz0_alignment, big);
            put_u32p(S, 0, false);
        } else if (kSplit<K>) {
            // MIO0.cs:64-81, Yay0.cs:63-78: magic, size, offsets of the code and the literal section (patched below)
            const char* magic = K == P_MIO0 ? "MIO0" : "Yay0";
            for (int i = 0; i < 4; i++) put_byte(S, uint8_t(magic[i]));
            put_u32p(S, uint32_t(n), big);
            put_u32p(S, 0, false);
            put_u32p(S, 0, false);
            // worst case n literal bytes / n code bytes: the layout of encode_lz.cu behind the (unused) finder tables
            S.codes = S.scratch + P.scratch_per_warp - 2 * (size_t(n) + 64);
            S.lits = S.codes + size_t(n) + 32;
            S.ncodes = S.nlits = 0;
            S.flag_base = S.pos;
        } else {
            put_byte(S, 'L'); put_byte(S, 'Z'); put_byte(S, 'S'); put_byte(S, 'S');
            put_u32p(S, uint32_t(n), true);
            put_u32p(S, 0, false);   // compressed size, patched below
            put_u32p(S, 0, false);
        }
        const uint64_t body_start = S.pos;
        // ---- tables: every head is 8192 positions back (behind the window)
        {
            const uint32_t far = uint32_t(0 - 8192) & 0xFFFFu;
            const uint32_t w = far | (far << 16);
            for (int i = lane; i < kBuckets / 2; i += 32) sts_u32(S.head + 4 * i, w);
            if (M)
                for (int i = lane; i < kBuckets / 2; i += 32) sts_u32(S.head2 + 4 * i, w);
        }
        __syncwarp();

        int plen = 0, pdist = 0;   // results of the previous step
        for (int base = 0; base < n; base += 32) {
            stage(S, base + 32 + S.look + 8);
            if (base && (base & 0x3FFF) == 0) {
                // heads that fell out of the window are parked 8192 positions back, so that their 16-bit age never wraps
                const uint32_t b16 = uint32_t(base) & 0xFFFFu;
                for (int i = lane; i < kBuckets; i += 32) {
                    const uint32_t e = lds_u16(S.head + 2 * i);
                    if (((b16 - e) & 0xFFFFu) > uint32_t(kWin)) sts_u16(S.head + 2 * i, (b16 - 8192u) & 0xFFFFu);
                    if (M) {
                        const uint32_t e2 = lds_u16(S.head2 + 2 * i);
                        if (((b16 - e2) & 0xFFFFu) > uint32_t(kWin)) sts_u16(S.head2 + 2 * i, (b16 - 8192u) & 0xFFFFu);
                    }
                }
                __syncwarp();
            }
            const int p = base + lane;
            const bool valid = p <= S.limit;
            // lanes inside a match that is already written are inserted but not searched (their results are never looked at)
            const bool searched = valid && (S.pending || lane >= S.cur_off);
            int best_len = 0, best_dist = 0;
            uint32_t h = 0xFFFFFFFFu, bucket = 0xFFFFFFFFu, ip = 0;   // ip: ring index of my position
            uint32_t hm = 0xFFFFFFFFu, bucket2 = 0xFFFFFFFFu;
            if (valid) {
                ip = didx(uint32_t(p) + S.skew);
                const uint32_t v4 = ring_u32_at(S, ip);
                h = ((v4 * 2654435761u) >> S.hash_shift) & S.hash_mask;   // ComputeHash, :288-299
                bucket = h & kBucketMask;
                if (M) {
                    hm = (((v4 & S.min_mask) * 2654435761u) >> 16) & 0xFFFFu;
                    bucket2 = hm & kBucketMask;
                }
            }
            uint32_t gm2b = 0, gm2h = 0, blink2 = 0;
            if (M) {
                gm2b = __match_any_sync(kFull, bucket2);
                gm2h = __match_any_sync(kFull, hm);
            }
            const uint32_t tag = h >> kBucketBits;
            const uint32_t lt = (1u << lane) - 1u;
            const uint32_t gmb = __match_any_sync(kFull, bucket);   // lanes of my bucket
            const uint32_t gmh = __match_any_sync(kFull, h);        // lanes with my hash value: the candidates inside this step
            uint32_t blink = 0;
            if (valid) {
                // ---- the bucket's chain before this step starts at its head
                const uint32_t e = lds_u16(S.head + 2 * bucket);
                const uint32_t dd = (uint32_t(p) - e) & 0xFFFFu;
                const bool head_ok = dd >= 1 && dd <= uint32_t(kWin) && int(dd) <= p;
                const uint32_t belowb = gmb & lt;
                blink = belowb ? uint32_t(lane - (31 - __clz(int(belowb)))) : (head_ok ? dd : 0u);
                // ---- chain walk (ChainMatches, :248-282): the candidates are the earlier positions with my hash value, nearest first
                const int best_possible = min(n - p, S.max_len);
                int attempts = S.max_chain;
                bool done = false;
                const int ring_cap = min(best_possible, S.look);   // what the ring can compare
                auto candidate = [&](int distance) {
                    attempts--;
                    // a candidate can only beat the best match so far if it also matches at offset best_len: one byte decides
                    // most of the later candidates of a chain (the result is the same: a longer match agrees on that byte)
                    const uint32_t ic = dwrap(ip + kData - uint32_t(distance));   // ring index of the candidate (distance <= 4096 < kData)
                    bool may_win = distance >= S.min_dist;
                    if (may_win && best_len != 0) {
                        if (K != P_LZ11 || best_len < ring_cap) may_win = lds_u8(S.data + dwrap(ip + uint32_t(best_len))) == lds_u8(S.data + dwrap(ic + uint32_t(best_len)));
                        else may_win = __ldg(S.src + p + best_len) == __ldg(S.src + p - distance + best_len);   // (best_len < best_possible <= n - p)
                    }
                    if (may_win) {
                        // the same distance as 32 positions earlier: that match's bytes behind the first 32 are equal here too
                        // CompatibilityMode cuts a match to its distance (LzChainMatchFinder.cs:304): comparing further cannot change the result (the
                        // reference compares best_possible bytes first, which makes long runs quadratic there)
                        const int cap = S.no_self_overlap ? min(best_possible, distance) : best_possible;
                        const int rcap = min(cap, ring_cap);
                        const int known = (distance == pdist && plen > 32) ? min(plen - 32, cap) : 0;
                        int l = prefix_len(S, ip, ic, rcap, min(known, rcap));
                        if (K == P_LZ11 && l == rcap && rcap < cap) l = extend_global(S.src + p, distance, max(known, rcap), cap);
                        if (l >= S.min_len && l > best_len) {
                            best_len = l;
                            best_dist = distance;
                            if (best_len == best_possible) done = true;
                        }
                    }
                    if (attempts <= 0) done = true;
                };
                uint32_t inl = searched ? gmh & lt : 0u;   // (a) inside the step
                done = !searched;
                while (inl && !done) {
                    const int k = 31 - __clz(int(inl));
                    inl &= ~(1u << k);
                    candidate(lane - k);
                }
                if (!done && head_ok && int(dd) <= S.max_dist) {   // (b) the ring: skip the nodes of my bucket with another tag
                    int distance = int(dd);
                    for (;;) {
                        const uint32_t nd = lds_u16(S.node + 2 * (uint32_t(p - distance) & kWinMask));
                        // three tag bits live in the node; a node that passes them is confirmed by hashing its four bytes again
                        if ((nd >> 13) == (tag & 7u) && (((ring_u32_at(S, dwrap(ip + kData - uint32_t(distance))) * 2654435761u) >> S.hash_shift) & S.hash_mask) == h) {
                            candidate(distance);
                            if (done) break;
                        }
                        const int bl = int(nd & 0x1FFFu);
                        if (bl == 0 || distance + bl > S.max_dist) break;
                        distance += bl;
                    }
                }
                if (M) {
                    // ---- the small-match table (MatchSearch, :236-244): only when the chain gave nothing; ONE candidate, the latest
                    // earlier position with my 16-bit hash of the first min_length bytes — whatever its distance
                    const uint32_t e2 = lds_u16(S.head2 + 2 * bucket2);
                    const uint32_t dd2 = (uint32_t(p) - e2) & 0xFFFFu;
                    const bool head2_ok = dd2 >= 1 && dd2 <= uint32_t(kWin) && int(dd2) <= p;
                    const uint32_t below2b = gm2b & lt;
                    blink2 = below2b ? uint32_t(lane - (31 - __clz(int(below2b)))) : (head2_ok ? dd2 : 0u);
                    if (searched && best_len == 0) {
                        int qd = 0;
                        const uint32_t below2h = gm2h & lt;
                        if (below2h) {
                            qd = lane - (31 - __clz(int(below2h)));
                        } else if (head2_ok && int(dd2) <= S.max_dist) {
                            int distance = int(dd2);
                            for (;;) {
                                const uint32_t nd = lds_u16(S.node2 + 2 * (uint32_t(p - distance) & kWinMask));
                                if ((nd >> 13) == ((hm >> kBucketBits) & 7u) &&
                                    ((((ring_u32_at(S, dwrap(ip + kData - uint32_t(distance))) & S.min_mask) * 2654435761u) >> 16) & 0xFFFFu) == hm) {
                                    qd = distance;
                                    break;
                                }
                                const int bl = int(nd & 0x1FFFu);
                                if (bl == 0 || distance + bl > S.max_dist) break;
                                distance += bl;
                            }
                        }
                        if (qd) {
                            const int distance = qd < S.min_dist ? S.min_dist : qd;
                            // (a raised distance that points in front of the buffer is no match: finder.cuh, DESIGN.md section 2, deviation 6)
                            if (distance <= S.max_dist && p - distance >= 0) {
                                const uint32_t ic = dwrap(ip + kData - uint32_t(distance));
                                const int cap = S.no_self_overlap ? min(best_possible, distance) : best_possible;
                                const int rcap = min(cap, ring_cap);
                                int l = prefix_len(S, ip, ic, rcap, 0);
                                if (K == P_LZ11 && l == rcap && rcap < cap) l = extend_global(S.src + p, distance, rcap, cap);
                                best_len = l;
                                best_dist = distance;
                            }
                        }
                    }
                }
            }
            __syncwarp();
            // ---- the step's positions enter the ring and the heads
            if (valid) {
                sts_u16(S.node + 2 * (uint32_t(p) & kWinMask), blink | ((tag & 7u) << 13));
                if ((gmb >> lane) <= 1u) sts_u16(S.head + 2 * bucket, uint32_t(p) & 0xFFFFu);   // the last lane of the bucket's group
                if (M) {
                    sts_u16(S.node2 + 2 * (uint32_t(p) & kWinMask), blink2 | (((hm >> kBucketBits) & 7u) << 13));
                    if ((gm2b >> lane) <= 1u) sts_u16(S.head2 + 2 * bucket2, uint32_t(p) & 0xFFFFu);
                }
            }
            __syncwarp();
            // ---- the token left pending at the end of the previous step: lazy test against this step's first result
            if (S.pending) {
                const int ln = __shfl_sync(kFull, best_len, 0), lk = __shfl_sync(kFull, plen, 31);
                S.pending = false;
                if (ln > lk) {
                    emit_step<K>(S, base - 32, plen, pdist, 0x80000000u, 0u);
                    S.forced = true;
                    S.cur_off = 0;
                } else {
                    emit_step<K>(S, base - 32, plen, pdist, 0u, 0x80000000u);
                    S.forced = false;
                    S.cur_off = lk - 1;
                }
            }
            // ---- parse + write this step
            uint32_t lit, mat;
            parse_step(S, base, best_len, lit, mat);
            emit_step<K>(S, base, best_len, best_dist, lit, mat);
            plen = best_len;
            pdist = best_dist;
        }
        if (K == P_LZSS) {
            const uint64_t save = S.pos;
            S.pos = 8;
            put_u32p(S, uint32_t(save - body_start), true);
            S.pos = save;
        }
        if (K == P_SMSR) {
            // the literal section follows the mask / code section
            __syncwarp();
            const uint64_t lit_off = S.pos;
            for (uint32_t i = lane; i < S.nlits; i += 32)
                if (lit_off + i < S.cap) S.out[lit_off + i] = S.lits[i];
            if (lit_off + S.nlits > S.cap) S.overflow = true;
            S.pos = 12;
            put_u32p(S, uint32_t(lit_off), true);
            S.pos = lit_off + S.nlits;
            __syncwarp();
        }
        if (kSplit<K>) {
            // the flag section is complete (every step wrote its groups, open ones included): codes and literals follow it
            __syncwarp();
            const uint64_t comp_off = body_start + ((S.ntok + 7u) >> 3), lit_off = comp_off + S.ncodes;
            for (uint32_t i = lane; i < S.ncodes; i += 32)
                if (comp_off + i < S.cap) S.out[comp_off + i] = S.codes[i];
            for (uint32_t i = lane; i < S.nlits; i += 32)
                if (lit_off + i < S.cap) S.out[lit_off + i] = S.lits[i];
            if (lit_off + S.nlits > S.cap) S.overflow = true;
            S.pos = 8;
            put_u32p(S, uint32_t(comp_off), big);
            put_u32p(S, uint32_t(lit_off), big);
            S.pos = lit_off + S.nlits;
            __syncwarp();
        }
        out_len = S.pos;
        if (S.overflow) status = AURORA_DST_TOO_SMALL;
    }
    const uint32_t ov = __ballot_sync(kFull, status != AURORA_OK);
    if (lane == 0) {
        P.out_len[idx] = out_len;
        P.status[idx] = ov ? (n64 > 0x7FFFFFF0ull ? AURORA_INVALID_ARGUMENT : AURORA_DST_TOO_SMALL) : AURORA_OK;
    }
    __syncwarp();
}

// the per-warp state from the batch parameters; `tables`: shared address of this warp's tables, `scratch`: its slice of the
// global scratch buffer (MIO0 / Yay0 sections).  (Also called by the CPU lane emulation of tests/simt.)
__device__ __forceinline__ void par_setup(ParState& S, const EncodeParams& P, uint32_t tables, uint8_t* scratch) {
    S.head = tables;
    S.node = tables + kBuckets * 2;
    S.data = S.node + kWin * 2;
    S.head2 = S.data + kData;
    S.node2 = S.head2 + kBuckets * 2;
    S.min_mask = 0xFFFFFFFFu >> ((4 - (P.min_length < 4 ? P.min_length : 4)) * 8);
    S.hash_shift = 32 - P.hash_bits;
    S.hash_mask = (1u << P.hash_bits) - 1u;
    S.max_chain = P.max_chain;
    S.lazy = P.lazy_threshold;
    S.min_len = P.min_length;
    S.max_len = P.max_length;
    S.look = P.max_length < kLook ? P.max_length : kLook;
    S.lz40 = P.format == AURORA_FMT_LZ40 || P.format == AURORA_FMT_LZ60;
    S.min_dist = P.min_distance;
    S.max_dist = P.max_distance;
    S.no_self_overlap = P.no_self_overlap != 0;
    S.blz = P.format == AURORA_FMT_BLZ;
    S.lz_n = P.lzss.max_distance - 1;
    S.lz_f = (1 << P.lzss.length_bits) - 1;
    S.lz_start = P.lzss.windows_start;
    S.lz_lbits = P.lzss.length_bits;
    S.scratch = scratch;
}

// ---- kernel
template <int K, bool M>
__global__ void __launch_bounds__(kParWarps<M> * 32, 1) encode_lz_par_kernel(const EncodeParams P) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int warp = threadIdx.x >> 5;
    ParState S;
    par_setup(S, P, smem_u32(smem) + uint32_t(warp) * kTablesPerWarp<M>, P.scratch + size_t(blockIdx.x * kParWarps<M> + warp) * P.scratch_per_warp);
    for (;;) {
        uint32_t t = 0;
        if (lane_id() == 0) t = atomicAdd(P.ticket, 1u);
        t = __shfl_sync(kFull, t, 0);
        if (t >= P.n) break;
        encode_stream_par<K, M>(P, t, S);
    }
}

template <int K, bool M>
cudaError_t launch_par_m(const EncodeParams& p, int blocks, cudaStream_t st) {
    const size_t smem = size_t(kParWarps<M>) * kTablesPerWarp<M>;
    static bool configured[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!configured[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(encode_lz_par_kernel<K, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
        if (e != cudaSuccess) return e;
        configured[dev & 63] = true;
    }
    encode_lz_par_kernel<K, M><<<blocks, kParWarps<M> * 32, smem, st>>>(p);
    return cudaGetLastError();
}

// the small-match table only exists at qualities >= 10 for formats whose shortest match is below 4 bytes (finder.cuh has_min)
template <int K>
cudaError_t launch_par(const EncodeParams& p, int blocks, cudaStream_t st) {
    return (p.use_min_table && p.min_length < 4) ? launch_par_m<K, true>(p, blocks, st) : launch_par_m<K, false>(p, blocks, st);
}

}  // namespace

// the formats / settings the parallel search reproduces exactly (everything else: encode_lz.cu)
bool encode_lz_par_supported(const EncodeParams& p) {
    const bool fmt = p.format == AURORA_FMT_LZ10 || p.format == AURORA_FMT_BLZ || p.format == AURORA_FMT_YAZ0 || p.format == AURORA_FMT_YAZ1 ||
                     p.format == AURORA_FMT_LZSS || p.format == AURORA_FMT_MIO0 || p.format == AURORA_FMT_YAY0 ||
                     p.format == AURORA_FMT_LZHUDSON || p.format == AURORA_FMT_SMSR00;
    const bool lz11 = p.format == AURORA_FMT_LZ11 || p.format == AURORA_FMT_LZ40 || p.format == AURORA_FMT_LZ60;   // any max_length
    // (one-byte matches with the small-match table, LZSS with min_length 1 from quality 10 on, parse differently from the
    //  reference here: the sequential replay writes its bytes)
    return (lz11 || (fmt && p.max_length <= kLook)) && p.hash_bits >= kBucketBits && p.hash_bits <= 24 && p.max_distance <= kWin && p.chain_bits >= 12 &&
           p.min_length >= 1 && p.min_distance >= 1 && !(p.use_min_table && p.min_length == 1);
}

int encode_lz_par_block_warps(const EncodeParams& p) {
    return (p.use_min_table && p.min_length < 4) ? kParWarps<true> : kParWarps<false>;
}

cudaError_t launch_encode_lz_par(const EncodeParams& p, int blocks, cudaStream_t st) {
    switch (p.format) {
        case AURORA_FMT_LZ10:
        case AURORA_FMT_BLZ: return launch_par<P_LZ10>(p, blocks, st);
        case AURORA_FMT_YAZ0:
        case AURORA_FMT_YAZ1: return launch_par<P_YAZ0>(p, blocks, st);
        case AURORA_FMT_LZSS: return launch_par<P_LZSS>(p, blocks, st);
        case AURORA_FMT_MIO0: return launch_par<P_MIO0>(p, blocks, st);
        case AURORA_FMT_YAY0: return launch_par<P_YAY0>(p, blocks, st);
        case AURORA_FMT_LZ11:
        case AURORA_FMT_LZ40:
        case AURORA_FMT_LZ60: return launch_par<P_LZ11>(p, blocks, st);
        case AURORA_FMT_LZHUDSON: return launch_par<P_HUDSON>(p, blocks, st);
        case AURORA_FMT_SMSR00: return launch_par<P_SMSR>(p, blocks, st);
        default: return cudaErrorNotSupported;
    }
}

}  // namespace aurora
