// wrappers.cu — the wrapper formats of AuroraLib.Compression.Nintendo (SURVEY.md 8f item 2): a header around one of the
// cores the kernels decode.  Every stream becomes one (ChunkLZ10: several independent) sub-stream of a core batch that runs
// on the device exactly like a direct call.  The header rule (wrap_resolve, wrap_chunk), the merge of the core results
// (wrap_merge) and the ChunkLZ10 redo selection (wrap_redo_chunk) are written once, above the "// ---- kernel" line, and are
// __host__ __device__: aurora_decode_batch resolves the headers on the host, aurora_decode_batch_device in
// wrap_resolve_kernel, one thread per stream.
//
// Reference semantics restated (paths under /root/reference/src/AuroraLib.Compression.Nintendo):
//   Nintendo/GCLZ.cs:39-53, Sega/CXLZ.cs:41-55, Nintendo/3DS-LZ.cs:37-50   magic + LZ10.Decompress / Compress
//   Sega/COMP.cs:39-53                                                    magic + LZ11
//   Nintendo/LZ77.cs:59-158   "LZ77", type byte, u24 size (u32 when 0): LZ10 / LZ11 headerless, or ChunkLZ10 = u16 end
//                             offsets + independent LZ10 streams of ChunkSize bytes each
//   Level5/Level5.cs:63-148   u32 LE (type | size << 3): OnlySave (stored) or LZ10 headerless; a payload starting with
//                             0x78 is zlib.  Huffman / RLE / zlib are not LZ hot-path codecs: NOT_SUPPORTED
//   Nintendo/LZOn.cs:41-80    "LZOn" 00 2F F1 71, BE size, BE compressed size, LZO headerless, ThrowIfMismatch(size)
//   Level5/Level5LZSS.cs:41-72 "SSZL", u32, compressed size, size, LZSS headerless with LZSS.Lzss0Properties
// The LZSS-property family (a fixed header + LZSS.DecompressHeaderless with DefaultProperties or Lzss0Properties) is table
// driven (family_of below): Sega/AKLZ.cs:43-56, Sega/LZ01.cs:47-82, Sega/LZSega.cs:49-67 (src/AuroraLib.Compression.Sega),
// Marvelous/FCMP.cs:43-59, Marvelous/IECP.cs:42-55, Konami/GCZ.cs:40-51, Specialized/MDB4.cs:41-80 (…-Extended).
// Two more LZSS wrappers do a little work around the core:
//   Specialized/ECD.cs:56-121 (…-Extended)  "ECD" + flag + plain size + compressed size + size (BE); the first `plain size`
//                             bytes are stored, the rest is LZSS(0x400, 0x42, 3, 0x3BE) headerless; or the whole payload is stored
//   Sega/LZ00.cs:50-203 (…Sega)  64-byte header with the decoded size and a key; the LZSS (Lzss0) body is XORed byte by byte
//                             with an LCG keystream: a device pass over the body (keystream.cu) before / after the LZSS kernel
#include <algorithm>
#include <cstring>
#include <vector>

#include "api_internal.hpp"
#include "common.cuh"
#include "size_peek.cuh"
#ifdef __CUDACC__
#include <cub/device/device_scan.cuh>
#endif

namespace aurora {

__host__ __device__ inline uint32_t le32(const uint8_t* p) { return uint32_t(p[0]) | (uint32_t(p[1]) << 8) | (uint32_t(p[2]) << 16) | (uint32_t(p[3]) << 24); }
__host__ __device__ inline uint32_t be32(const uint8_t* p) { return (uint32_t(p[0]) << 24) | (uint32_t(p[1]) << 16) | (uint32_t(p[2]) << 8) | p[3]; }
__host__ __device__ inline uint64_t umin(uint64_t a, uint64_t b) { return a < b ? a : b; }
__host__ __device__ inline const char* lzon_magic() { return "LZOn\0\x2F\xF1\x71"; }   // 8 bytes

constexpr uint64_t kParseHeader = ~0ull;   // raw size "none": the core parses its own header

// LZSS-property family: identifier, header bytes that are READ (a short stream is END_OF_STREAM), bytes skipped by a seek
// after them, where the decoded size sits, and which LzProperties the body uses.  A switch rather than a table: device code
// cannot read a host array.
struct Family {
    int format;
    const char* magic;
    uint32_t magic_len, read_len, skip_len, size_off;
    bool size_big, lzss0;
};
__host__ __device__ inline bool family_of(int format, Family& f) {
    switch (format) {
        case AURORA_FMT_AKLZ: f = Family{format, "AKLZ~?Qd=\xCC\xCC\xCD", 12, 16, 0, 12, true, false}; return true;
        case AURORA_FMT_LZ01: f = Family{format, "LZ01", 4, 16, 0, 8, false, true}; return true;
        case AURORA_FMT_FCMP: f = Family{format, "FCMP", 4, 12, 0, 4, false, true}; return true;
        case AURORA_FMT_IECP: f = Family{format, "IECP", 4, 8, 0, 4, false, true}; return true;
        case AURORA_FMT_MDB4: f = Family{format, "MDB4", 4, 16, 16, 8, false, false}; return true;
        case AURORA_FMT_LZSEGA: f = Family{format, "", 0, 8, 0, 4, false, false}; return true;
        case AURORA_FMT_GCZ: f = Family{format, "", 0, 4, 0, 0, false, true}; return true;
        // LZ00.cs:56-63: magic, length, 8 skipped (a seek), 32-byte name, size, key are READ up to byte 56; 8 more are skipped
        case AURORA_FMT_LZ00: f = Family{format, "LZ00", 4, 56, 8, 48, false, true}; return true;
    }
    return false;
}

// the one core sub-stream of a wrapped stream, or one ChunkLZ10 chunk
struct WrapSub {
    int core;           // AURORA_FMT_LZ10 / LZ11 / LZSS / LZO; 0: no sub-stream (header error, stored payload)
    uint64_t off, len;  // source bytes, relative to the wrapped stream
    uint64_t doff;      // destination offset inside the wrapped stream's slot
    uint64_t raw;       // kParseHeader or the decoded size of a headerless body
    uint32_t key;       // LZ00: keystream key of the body
};

struct WrapPlan {
    int status;              // header-level result (the core statuses are merged in afterwards)
    uint64_t consumed;       // source position when a header-level error was raised
    uint64_t out_len;        // bytes of a stored payload
    uint64_t expect;         // LZ77 chunked / LZOn / SDPC: the size the header promises
    uint64_t end_consumed;   // LZ77 chunked: source position after the last chunk
    uint64_t chunks, table;  // LZ77 chunked: number of chunks (0: not chunked), position of their u16 end-offset table
    // bytes at the start of the destination slot that no core writes (stored payloads, ECD's plain prefix): copy_len bytes
    // from source position copy_off, then fill_len bytes of 0xFF
    uint64_t copy_off, copy_len, fill_len;
};

// Magic check with the stream semantics of MatchThrow: short stream -> END_OF_STREAM (position at the end), wrong
// bytes -> INVALID_IDENTIFIER (position after the identifier)
__host__ __device__ inline bool match_throw(WrapPlan& pl, const uint8_t* p, uint64_t len, const char* magic, uint64_t k) {
    if (len < k) {
        pl.status = AURORA_END_OF_STREAM;
        pl.consumed = len;
        return false;
    }
    for (uint64_t j = 0; j < k; j++) {
        if (p[j] != uint8_t(magic[j])) {
            pl.status = AURORA_INVALID_IDENTIFIER;
            pl.consumed = k;
            return false;
        }
    }
    return true;
}

__host__ __device__ inline void eos(WrapPlan& pl, uint64_t len) {
    pl.status = AURORA_END_OF_STREAM;
    pl.consumed = len;
}

// The header rule: the plan of one wrapped stream of `len` bytes with a destination of `cap` bytes, and its sub-stream.
// ChunkLZ10 leaves `sub` empty and sets pl.chunks: the chunks are enumerated with wrap_chunk.
__host__ __device__ inline void wrap_resolve(int format, const uint8_t* p, uint64_t len, uint64_t cap, WrapPlan& pl, WrapSub& sub) {
    pl = WrapPlan{AURORA_OK, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    sub = WrapSub{0, 0, 0, 0, 0, 0u};
    auto one = [&](int core, uint64_t off, uint64_t raw) { sub = WrapSub{core, off, len - off, 0, raw, 0u}; };
    switch (format) {
        case AURORA_FMT_GCLZ:
            if (match_throw(pl, p, len, "GCLZ", 4)) one(AURORA_FMT_LZ10, 4, kParseHeader);
            break;
        case AURORA_FMT_CXLZ:
            if (match_throw(pl, p, len, "CXLZ", 4)) one(AURORA_FMT_LZ10, 4, kParseHeader);
            break;
        case AURORA_FMT_COMP:
            if (match_throw(pl, p, len, "COMP", 4)) one(AURORA_FMT_LZ11, 4, kParseHeader);
            break;
        case AURORA_FMT_LZ_3DS:
            if (match_throw(pl, p, len, "3DS-LZ\r\n", 8)) one(AURORA_FMT_LZ10, 8, kParseHeader);
            break;
        case AURORA_FMT_LZON:
            if (!match_throw(pl, p, len, lzon_magic(), 8)) break;
            if (len < 16) { eos(pl, len); break; }
            pl.expect = be32(p + 8);
            one(AURORA_FMT_LZO, 16, kParseHeader);
            break;
        case AURORA_FMT_SDPC: {   // -Extended/Specialized/SDPC.cs:43-56: SetLength(size) up front, overshoot check afterwards
            if (!match_throw(pl, p, len, "SDPC", 4)) break;
            if (len < 8) { eos(pl, len); break; }
            pl.expect = le32(p + 4);
            if (pl.expect > cap) { pl.status = AURORA_DST_TOO_SMALL; pl.consumed = 8; break; }
            one(AURORA_FMT_LZO, 8, kParseHeader);
            break;
        }
        case AURORA_FMT_LEVEL5_LZSS:
            if (!match_throw(pl, p, len, "SSZL", 4)) break;
            if (len < 16) { eos(pl, len); break; }
            one(AURORA_FMT_LZSS, 16, le32(p + 12));
            break;
        case AURORA_FMT_LEVEL5: {
            if (len < 5) { eos(pl, len); break; }   // ReadUInt32 + Peek<byte>()
            const uint32_t v = le32(p);
            if (p[4] == 0x78) { pl.status = AURORA_NOT_SUPPORTED; pl.consumed = 4; break; }   // zlib payload
            const uint32_t type = v & 7, size = v >> 3;
            if (type == 0) {   // OnlySave: ReadExactly + Write
                if (uint64_t(size) > len - 4) { eos(pl, len); break; }
                pl.copy_off = 4;
                pl.copy_len = umin(size, cap);
                pl.out_len = size;
                pl.consumed = 4 + uint64_t(size);
                if (size > cap) pl.status = AURORA_DST_TOO_SMALL;
            } else if (type == 1) {
                one(AURORA_FMT_LZ10, 4, size);
            } else {
                pl.status = AURORA_NOT_SUPPORTED;
                pl.consumed = 4;
            }
            break;
        }
        case AURORA_FMT_LZ77: {
            if (!match_throw(pl, p, len, "LZ77", 4)) break;
            if (len < 8) { eos(pl, len); break; }   // type byte + u24
            const uint8_t type = p[4];
            uint64_t pos = 8;
            uint32_t size = uint32_t(p[5]) | (uint32_t(p[6]) << 8) | (uint32_t(p[7]) << 16);
            if (size == 0) {
                if (len < 12) { eos(pl, len); break; }
                size = le32(p + 8);
                pos = 12;
            }
            if (type == 0x10 || type == 0x11) {
                // type byte + size are exactly an LZ10 / LZ11 header: DecompressHeaderless(size) == Decompress from offset 4
                one(type == 0x10 ? AURORA_FMT_LZ10 : AURORA_FMT_LZ11, 4, kParseHeader);
            } else if (type == 0xF7) {
                // u16 end offsets until one of them, added to the position behind it, is the end of the stream
                const uint64_t table = pos;
                uint64_t count = 0, end = 0;
                for (;;) {
                    if (pos + 2 > len) { eos(pl, len); break; }
                    end = uint32_t(p[pos]) | (uint32_t(p[pos + 1]) << 8);
                    pos += 2;
                    count++;
                    if (end + pos == len) break;
                }
                if (pl.status != AURORA_OK) break;
                pl.expect = size;
                pl.table = table;
                pl.chunks = count;
                pl.end_consumed = pos + end;
            } else {
                pl.status = AURORA_NOT_SUPPORTED;   // HUF20 / RLE30 sub-types, undefined values
                pl.consumed = pos;
            }
            break;
        }
        case AURORA_FMT_ECD: {   // ECD.cs:56-86
            if (!match_throw(pl, p, len, "ECD", 3)) break;
            if (len < 16) { eos(pl, len); break; }   // ReadByte() is -1 at the end, the three ReadUInt32 throw
            const bool compressed = p[3] == 1;
            const uint64_t plain = be32(p + 4), size = be32(p + 12);
            if (!compressed) {   // source.CopyTo(destination)
                const uint64_t rest = len - 16;
                pl.copy_off = 16;
                pl.copy_len = umin(rest, cap);
                pl.out_len = rest;
                pl.consumed = len;
                if (rest > cap) pl.status = AURORA_DST_TOO_SMALL;
                break;
            }
            // destination.WriteByte((byte)source.ReadByte()) plain times: past the end of the source that is 0xFF; a
            // fixed-size destination refuses the first byte past its capacity
            const uint64_t have = umin(plain, len - 16), fits = umin(plain, cap);
            pl.copy_off = 16;
            pl.copy_len = umin(have, fits);
            pl.fill_len = fits > have ? fits - have : 0;
            if (plain > cap) {
                pl.status = AURORA_DST_TOO_SMALL;
                pl.out_len = cap;
                pl.consumed = 16 + umin(cap, len - 16);
                break;
            }
            pl.out_len = plain;
            sub = WrapSub{AURORA_FMT_LZSS, 16 + have, len - 16 - have, plain, uint64_t(uint32_t(size - plain)), 0u};
            break;
        }
        default: {
            Family f{};
            if (!family_of(format, f)) { pl.status = AURORA_INVALID_ARGUMENT; break; }
            if (f.magic_len && !match_throw(pl, p, len, f.magic, f.magic_len)) break;
            if (len < f.read_len) { eos(pl, len); break; }
            const uint32_t size = f.size_big ? be32(p + f.size_off) : le32(p + f.size_off);
            one(AURORA_FMT_LZSS, umin(f.read_len + f.skip_len, len), size);   // Skip() is a seek: it may pass the end
            if (format == AURORA_FMT_LZ00) sub.key = le32(p + 52);
            break;
        }
    }
}

// ChunkLZ10 chunk k of a stream whose plan has chunks; doff is the decoded size of chunks 0 .. k-1 (every chunk is a complete
// LZ10 stream: its header gives the size that places the next one, wrap_chunk_size)
__host__ __device__ inline WrapSub wrap_chunk(const uint8_t* p, uint64_t len, const WrapPlan& pl, uint64_t k, uint64_t doff) {
    const uint64_t body = pl.table + 2 * pl.chunks;
    const uint64_t start = k == 0 ? body : body + (uint32_t(p[pl.table + 2 * k - 2]) | (uint32_t(p[pl.table + 2 * k - 1]) << 8));
    return WrapSub{AURORA_FMT_LZ10, umin(start, len), start <= len ? len - start : 0, doff, kParseHeader, 0u};
}
__host__ __device__ inline uint64_t wrap_chunk_size(const uint8_t* p, const WrapSub& c) {
    uint64_t size;   // 0 when the chunk's header does not parse
    core_decoded_size(AURORA_FMT_LZ10, AURORA_ENDIAN_DEFAULT, p + c.off, c.len, &size);
    return size;
}

// The merge rule: the stream's out_len / consumed / status from its plan and the core results of its sub-streams (sub[k],
// r_*[k] for k < pl.chunks, or the one sub-stream sub[0]).
__host__ __device__ inline void wrap_merge(int format, const WrapPlan& pl, const WrapSub* sub, const uint64_t* r_out, const uint64_t* r_cons,
                                           const int32_t* r_st, uint64_t& ol, uint64_t& cs, int& st) {
    ol = pl.out_len;
    cs = pl.consumed;
    st = pl.status;
    if (st != AURORA_OK) return;
    if (pl.chunks) {
        // chunks decode one after the other: the first failure ends the stream
        for (uint64_t k = 0; k < pl.chunks; k++) {
            ol = sub[k].doff + r_out[k];
            cs = sub[k].off + r_cons[k];
            if (r_st[k] != AURORA_OK) { st = r_st[k]; return; }
            // a chunk that decodes to a size other than its header's would shift the following ones
            if (k + 1 < pl.chunks && sub[k + 1].doff != ol) { st = AURORA_INVALID_DATA; return; }
        }
        cs = pl.end_consumed;
        if (ol > pl.expect) st = AURORA_SIZE_MISMATCH;
    } else if (sub[0].core) {
        ol = sub[0].doff + r_out[0];   // doff: ECD's plain bytes in front of the LZSS output
        cs = sub[0].off + r_cons[0];
        st = r_st[0];
        // ThrowIfMismatch runs before the destination's overflow is noticed
        if (format == AURORA_FMT_LZON && (st == AURORA_OK || st == AURORA_DST_TOO_SMALL) && ol != pl.expect) st = AURORA_SIZE_MISMATCH;
        if (format == AURORA_FMT_SDPC && (st == AURORA_OK || st == AURORA_DST_TOO_SMALL) && ol > pl.expect) st = AURORA_SIZE_MISMATCH;
    }
}

// ChunkLZ10 on corrupt input: the reference decodes the chunks one after the other and stops at the first failure, so the
// bytes a failing chunk writes past its own size (an overshooting last match: SIZE_MISMATCH) are the last thing its
// destination sees.  All chunks run at once and the next chunk writes the same bytes, so that chunk is decoded once more,
// alone, afterwards, and its bytes win deterministically.  The chunk to redo (-1: none), from the chunks' core statuses.
__host__ __device__ inline int64_t wrap_redo_chunk(const WrapPlan& pl, const int32_t* r_st) {
    if (pl.status != AURORA_OK) return -1;
    for (uint64_t k = 0; k < pl.chunks; k++) {
        if (r_st[k] == AURORA_OK) continue;
        return r_st[k] == AURORA_SIZE_MISMATCH && k + 1 < pl.chunks ? int64_t(k) : -1;
    }
    return -1;
}

// ---- kernel
namespace {

// the cores each wrapper format runs: `core` for every sub-stream, LZ77 also `core2` (LZ11) for its type-0x11 streams;
// `headerless`: the bodies are DecompressHeaderless (raw size in the upper half of the capacity word)
struct WrapCores {
    int core, core2;
    bool headerless;
};
WrapCores wrap_cores(int format) {
    switch (format) {
        case AURORA_FMT_GCLZ: case AURORA_FMT_CXLZ: case AURORA_FMT_LZ_3DS: return {AURORA_FMT_LZ10, 0, false};
        case AURORA_FMT_COMP: return {AURORA_FMT_LZ11, 0, false};
        case AURORA_FMT_LZ77: return {AURORA_FMT_LZ10, AURORA_FMT_LZ11, false};
        case AURORA_FMT_LEVEL5: return {AURORA_FMT_LZ10, 0, true};
        case AURORA_FMT_LZON: case AURORA_FMT_SDPC: return {AURORA_FMT_LZO, 0, false};
        default: return {AURORA_FMT_LZSS, 0, true};   // Level5LZSS, ECD, the LZSS-property family
    }
}

void family_props(const Family& f, aurora_lz_props* lz) {
    if (f.lzss0) aurora_lz_props_window(lz, 0x1000, 0xF + 3, 3, 0xFEE, 1);   // LZSS.Lzss0Properties (LZSS.cs:34)
    else aurora_lz_props_bits(lz, 12, 4, 2);                                 // LZSS.DefaultProperties (LZSS.cs:33)
}

// the caller's options with the LzProperties the format fixes
aurora_codec_opts wrap_core_opts(int format, const aurora_codec_opts* opts) {
    aurora_codec_opts o;
    if (opts) o = *opts;
    else aurora_codec_opts_init(&o);
    Family f{};
    if (format == AURORA_FMT_LEVEL5_LZSS) aurora_lz_props_window(&o.lzss, 0x1000, 0xF + 3, 3, 0xFEE, 1);   // LZSS.Lzss0Properties
    if (family_of(format, f)) family_props(f, &o.lzss);
    if (format == AURORA_FMT_ECD) aurora_lz_props_window(&o.lzss, 0x400, 0x42, 3, 0x3BE, 1);   // ECD.cs:18
    return o;
}

// one core launch's descriptors, in the kernels' convention (DecodeParams)
struct WrapSlots {
    uint64_t *src_off, *src_len, *dst_off, *dst_cap, *out_len, *consumed;
    int32_t* status;
    uint32_t* key;   // LZ00 only
};

// slot j of S for sub-stream s of a stream at (src_off, dst_off, cap): a sub-stream of another core is an empty stream
// (length 0, capacity 0) that fails at once and that the merge ignores.  The offsets do not depend on the core, so slot sets
// of two cores may share their offset arrays.
__device__ void put_slot(const WrapSlots& S, uint64_t j, const WrapSub& s, int core, bool headerless, uint64_t src_off, uint64_t dst_off,
                         uint64_t cap) {
    const bool use = s.core == core;
    S.src_off[j] = src_off + s.off;
    S.dst_off[j] = dst_off + umin(s.doff, cap);
    S.src_len[j] = use ? s.len : 0;
    // (ChunkLZ10: the capacity windows of one file's chunks overlap — every chunk may write up to the end of the file's slot,
    //  like the reference's single destination stream)
    uint64_t c = use && s.doff < cap ? cap - s.doff : 0;
    if (headerless) c = (use ? s.raw << 32 : 0) | umin(c, 0xFFFFFFFFull);   // DecodeParams::headerless
    S.dst_cap[j] = c;
    if (S.key) S.key[j] = s.key;
}

__global__ void wrap_resolve_kernel(int format, const uint8_t* src, const uint64_t* src_off, const uint64_t* src_len, const uint64_t* dst_off,
                                    const uint64_t* dst_cap, uint32_t n, WrapPlan* plans, WrapSub* subs, uint64_t* chunks, WrapSlots A,
                                    int core, int headerless) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    WrapPlan pl;
    WrapSub s;
    wrap_resolve(format, src + src_off[i], src_len[i], dst_cap[i], pl, s);
    plans[i] = pl;
    subs[i] = s;
    if (chunks) {   // LZ77: chunk counts for the scan (entry n stays 0, so the scan's entry n is the total)
        chunks[i] = pl.chunks;
        if (i == 0) chunks[n] = 0;
    }
    if (A.src_off) put_slot(A, i, s, core, headerless != 0, src_off[i], dst_off[i], dst_cap[i]);
}

// LZ77: stream slot i of both cores, then the chunk slots of stream i behind the n stream slots, at n + base[i]
__global__ void wrap_chunk_fill_kernel(const uint8_t* src, const uint64_t* src_off, const uint64_t* src_len, const uint64_t* dst_off,
                                       const uint64_t* dst_cap, uint32_t n, const WrapPlan* plans, const WrapSub* subs,
                                       const uint64_t* base, WrapSlots A, WrapSlots B, WrapSub* chunk_subs) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const WrapSub s = subs[i];
    const uint64_t so = src_off[i], dof = dst_off[i], cap = dst_cap[i];
    put_slot(A, i, s, AURORA_FMT_LZ10, false, so, dof, cap);
    put_slot(B, i, s, AURORA_FMT_LZ11, false, so, dof, cap);
    const WrapPlan pl = plans[i];
    const uint8_t* p = src + so;
    uint64_t doff = 0;
    for (uint64_t k = 0; k < pl.chunks; k++) {
        const WrapSub c = wrap_chunk(p, src_len[i], pl, k, doff);
        chunk_subs[base[i] + k] = c;
        put_slot(A, n + base[i] + k, c, AURORA_FMT_LZ10, false, so, dof, cap);
        doff += wrap_chunk_size(p, c);
    }
}

// LZ77: the redo launch's chunk slots — the chunk wrap_redo_chunk picks keeps its length and capacity, every other one is empty
__global__ void wrap_redo_select_kernel(uint32_t n, const WrapPlan* plans, const uint64_t* base, WrapSlots A, WrapSlots R) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const WrapPlan pl = plans[i];
    const uint64_t j0 = base[i];
    const int64_t r = wrap_redo_chunk(pl, A.status + n + j0);
    for (uint64_t k = 0; k < pl.chunks; k++) {
        const bool keep = int64_t(k) == r;
        R.src_len[j0 + k] = keep ? A.src_len[n + j0 + k] : 0;
        R.dst_cap[j0 + k] = keep ? A.dst_cap[n + j0 + k] : 0;
    }
}

// warp-cooperative copy in words of T: bytes up to T's alignment of d, then words, then the tail (s and d must have the same
// address modulo sizeof(T))
template <typename T>
__device__ void warp_copy(uint8_t* d, const uint8_t* s, uint64_t len, uint32_t lane) {
    const uint64_t head = umin((sizeof(T) - (reinterpret_cast<uintptr_t>(d) & (sizeof(T) - 1))) & (sizeof(T) - 1), len);
    for (uint64_t j = lane; j < head; j += 32) d[j] = s[j];
    const uint64_t words = (len - head) / sizeof(T);
    T* dw = reinterpret_cast<T*>(d + head);
    const T* sw = reinterpret_cast<const T*>(s + head);
    for (uint64_t j = lane; j < words; j += 32) dw[j] = sw[j];
    for (uint64_t j = head + words * sizeof(T) + lane; j < len; j += 32) d[j] = s[j];
}

// stored payloads (Level5 OnlySave, ECD stored) and ECD's plain prefix and its 0xFF fill: one warp per stream, 16-byte
// accesses when source and destination share their address modulo 16 (else 8, 4 or 1 byte)
__global__ void wrap_store_kernel(const uint8_t* src, const uint64_t* src_off, uint8_t* dst, const uint64_t* dst_off, const WrapPlan* plans,
                                  uint32_t n) {
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n) return;
    const uint64_t copy_off = plans[w].copy_off, copy_len = plans[w].copy_len, fill_len = plans[w].fill_len;
    uint8_t* d = dst + dst_off[w];
    if (copy_len) {
        const uint8_t* s = src + src_off[w] + copy_off;
        const uintptr_t mis = reinterpret_cast<uintptr_t>(d) ^ reinterpret_cast<uintptr_t>(s);
        if ((mis & 15) == 0) warp_copy<uint4>(d, s, copy_len, lane);
        else if ((mis & 7) == 0) warp_copy<uint2>(d, s, copy_len, lane);
        else if ((mis & 3) == 0) warp_copy<uint32_t>(d, s, copy_len, lane);
        else warp_copy<uint8_t>(d, s, copy_len, lane);
    }
    for (uint64_t j = lane; j < fill_len; j += 32) d[copy_len + j] = 0xFF;
}

__global__ void wrap_merge_kernel(int format, uint32_t n, const WrapPlan* plans, const WrapSub* subs, const WrapSub* chunk_subs,
                                  const uint64_t* base, WrapSlots A, WrapSlots B, int core2, uint64_t* out_len, uint64_t* consumed,
                                  int32_t* status) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const WrapPlan pl = plans[i];
    uint64_t ol, cs;
    int st;
    if (pl.chunks) {
        const uint64_t j = n + base[i];
        wrap_merge(format, pl, chunk_subs + base[i], A.out_len + j, A.consumed + j, A.status + j, ol, cs, st);
    } else {
        const WrapSlots& R = core2 && subs[i].core == core2 ? B : A;
        wrap_merge(format, pl, subs + i, R.out_len + i, R.consumed + i, R.status + i, ol, cs, st);
    }
    if (out_len) out_len[i] = ol;
    if (consumed) consumed[i] = cs;
    status[i] = st;
}

// carve 16-byte aligned arrays out of one scratch block
struct Carve {
    uint8_t* p;
    template <typename T>
    T* take(uint64_t count) {
        T* r = reinterpret_cast<T*>(p);
        p += (count * sizeof(T) + 15) & ~uint64_t(15);
        return r;
    }
};
uint64_t slot_bytes(uint64_t m) { return 6 * ((m * 8 + 15) & ~15ull) + 2 * ((m * 4 + 15) & ~15ull); }
WrapSlots take_slots(Carve& c, uint64_t m) {
    WrapSlots S;
    S.src_off = c.take<uint64_t>(m);
    S.src_len = c.take<uint64_t>(m);
    S.dst_off = c.take<uint64_t>(m);
    S.dst_cap = c.take<uint64_t>(m);
    S.out_len = c.take<uint64_t>(m);
    S.consumed = c.take<uint64_t>(m);
    S.status = c.take<int32_t>(m);
    S.key = c.take<uint32_t>(m);
    return S;
}

#define WRAP_TRY(expr)                                   \
    do {                                                 \
        const cudaError_t e_ = (expr);                   \
        if (e_ != cudaSuccess) return e_;                \
    } while (0)

}  // namespace

bool is_wrapper_format(int f) { return f >= AURORA_FMT_GCLZ && f <= AURORA_FMT_LZ00; }

int wrapped_decode_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                         const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                         const uint64_t* dst_cap, uint64_t* out_len, uint64_t* consumed, int32_t* status) {
    std::vector<WrapPlan> plans(n);
    std::vector<WrapSub> subs;      // every stream's sub-streams, stream after stream
    std::vector<size_t> owner, first(n);
    subs.reserve(n);
    owner.reserve(n);
    for (size_t i = 0; i < n; i++) {
        const uint8_t* p = src_base + src_off[i];
        WrapSub s;
        wrap_resolve(format, p, src_len[i], dst_cap[i], plans[i], s);
        first[i] = subs.size();
        uint64_t doff = 0;
        for (uint64_t k = 0; k < plans[i].chunks; k++) {
            subs.push_back(wrap_chunk(p, src_len[i], plans[i], k, doff));
            owner.push_back(i);
            doff += wrap_chunk_size(p, subs.back());
        }
        if (s.core) {
            subs.push_back(s);
            owner.push_back(i);
        }
    }

    // one core batch per core format
    std::vector<uint64_t> r_out(subs.size(), 0), r_cons(subs.size(), 0);
    std::vector<int32_t> r_st(subs.size(), AURORA_OK);
    const aurora_codec_opts o = wrap_core_opts(format, opts);
    for (int key = 0; key < 8; key++) {   // one batch per (core format, headerless or not)
        static const int kCores[4] = {AURORA_FMT_LZ10, AURORA_FMT_LZ11, AURORA_FMT_LZSS, AURORA_FMT_LZO};
        const int core = kCores[key >> 1];
        const bool want_raw = (key & 1) != 0;
        std::vector<size_t> idx;
        for (size_t k = 0; k < subs.size(); k++)
            if (subs[k].core == core && (subs[k].raw != kParseHeader) == want_raw) idx.push_back(k);
        if (idx.empty()) continue;
        const size_t m = idx.size();
        std::vector<uint64_t> so(m), sl(m), dof(m), dc(m), raw(m), ol(m), cs(m);
        std::vector<int32_t> st(m);
        std::vector<uint32_t> keys;
        if (format == AURORA_FMT_LZ00) keys.resize(m);
        for (size_t j = 0; j < m; j++) {
            const WrapSub& s = subs[idx[j]];
            const size_t i = owner[idx[j]];
            so[j] = src_off[i] + s.off;
            sl[j] = s.len;
            const uint64_t cap = dst_cap[i];
            dof[j] = dst_off[i] + std::min(s.doff, cap);
            dc[j] = s.doff < cap ? cap - s.doff : 0;
            // (ChunkLZ10: the capacity windows of one file's chunks overlap — every chunk may write up to the end of the
            //  file's slot, like the reference's single destination stream; decode_core_batch keeps such streams on one device)
            raw[j] = s.raw;
            if (!keys.empty()) keys[j] = s.key;
        }
        const int rc = decode_core_batch(ctx, core, &o, m, src_base, so.data(), sl.data(), dst_base, dof.data(), dc.data(),
                                         want_raw ? raw.data() : nullptr, ol.data(), cs.data(), st.data(),
                                         keys.empty() ? nullptr : keys.data(), /*exact=*/true);
        if (rc != AURORA_OK) return rc;
        for (size_t j = 0; j < m; j++) {
            r_out[idx[j]] = ol[j];
            r_cons[idx[j]] = cs[j];
            r_st[idx[j]] = st[j];
        }
    }

    // ChunkLZ10: the failing chunks wrap_redo_chunk picks, decoded once more, alone
    if (format == AURORA_FMT_LZ77) {
        std::vector<size_t> redo;
        for (size_t i = 0; i < n; i++) {
            const int64_t k = wrap_redo_chunk(plans[i], r_st.data() + first[i]);
            if (k >= 0) redo.push_back(first[i] + size_t(k));
        }
        if (!redo.empty()) {
            const size_t m = redo.size();
            std::vector<uint64_t> so(m), sl(m), dof(m), dc(m), ol(m), cs(m);
            std::vector<int32_t> st(m);
            for (size_t j = 0; j < m; j++) {
                const WrapSub& s = subs[redo[j]];
                const size_t i = owner[redo[j]];
                const uint64_t cap = dst_cap[i];
                so[j] = src_off[i] + s.off;
                sl[j] = s.len;
                dof[j] = dst_off[i] + std::min(s.doff, cap);
                dc[j] = s.doff < cap ? cap - s.doff : 0;
            }
            const int rc = decode_core_batch(ctx, AURORA_FMT_LZ10, &o, m, src_base, so.data(), sl.data(), dst_base, dof.data(), dc.data(),
                                             nullptr, ol.data(), cs.data(), st.data(), nullptr, /*exact=*/true);
            if (rc != AURORA_OK) return rc;
        }
    }

    // stored bytes are written after the core batches: their device-to-host copies of a contiguous destination span also
    // cover the gaps between their streams
    const WrapSub none{};
    for (size_t i = 0; i < n; i++) {
        const WrapPlan& pl = plans[i];
        const size_t q = first[i], q_end = i + 1 < n ? first[i + 1] : subs.size();
        uint64_t ol, cs;
        int st;
        wrap_merge(format, pl, q < q_end ? subs.data() + q : &none, r_out.data() + q, r_cons.data() + q, r_st.data() + q, ol, cs, st);
        if (pl.copy_len) std::memcpy(dst_base + dst_off[i], src_base + src_off[i] + pl.copy_off, size_t(pl.copy_len));
        if (pl.fill_len) std::memset(dst_base + dst_off[i] + pl.copy_len, 0xFF, size_t(pl.fill_len));
        if (out_len) out_len[i] = ol;
        if (consumed) consumed[i] = cs;
        status[i] = st;
    }
    return AURORA_OK;
}

cudaError_t wrapped_decode_batch_device(int format, const aurora_codec_opts* opts, size_t n, const uint8_t* d_src_base, uint64_t src_total,
                                        const uint64_t* d_src_off, const uint64_t* d_src_len, uint8_t* d_dst_base,
                                        const uint64_t* d_dst_off, const uint64_t* d_dst_cap, uint64_t* d_out_len,
                                        uint64_t* d_consumed, int32_t* d_status, WrapScratch& scr, unsigned int* ticket, int sm_count,
                                        cudaStream_t st, uint64_t* launches) {
    const WrapCores cores = wrap_cores(format);
    const aurora_codec_opts o = wrap_core_opts(format, opts);
    const bool lz77 = format == AURORA_FMT_LZ77;
    const uint32_t N = uint32_t(n);
    const unsigned grid = (N + 127) / 128;

    // per-stream scratch: plans, sub-streams, LZ77's chunk counts and their exclusive scan, the scan's temporary storage
    size_t scan_bytes = 0;
    if (lz77) WRAP_TRY(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, static_cast<uint64_t*>(nullptr), static_cast<uint64_t*>(nullptr), n + 1, st));
    const uint64_t per_stream = ((n * sizeof(WrapPlan) + 15) & ~15ull) + ((n * sizeof(WrapSub) + 15) & ~15ull) + 2 * (((n + 1) * 8 + 15) & ~15ull) + scan_bytes;
    WRAP_TRY(scr.plans.reserve(per_stream));
    Carve cp{static_cast<uint8_t*>(scr.plans.p)};
    WrapPlan* plans = cp.take<WrapPlan>(n);
    WrapSub* subs = cp.take<WrapSub>(n);
    uint64_t* counts = cp.take<uint64_t>(n + 1);
    uint64_t* base = cp.take<uint64_t>(n + 1);
    void* scan_tmp = cp.p;

    WrapSlots A{}, B{}, R{};
    WrapSub* chunk_subs = nullptr;
    uint64_t m = n;
    if (!lz77) {   // the stream slots are the whole launch: the resolve pass writes them
        WRAP_TRY(scr.slots.reserve(slot_bytes(n)));
        Carve cs{static_cast<uint8_t*>(scr.slots.p)};
        A = take_slots(cs, n);
        if (format != AURORA_FMT_LZ00) A.key = nullptr;
    }
    wrap_resolve_kernel<<<grid, 128, 0, st>>>(format, d_src_base, d_src_off, d_src_len, d_dst_off, d_dst_cap, N, plans, subs,
                                              lz77 ? counts : nullptr, A, cores.core, cores.headerless);
    WRAP_TRY(cudaGetLastError());
    ++*launches;
    if (lz77) {
        // the chunk slots follow the n stream slots; their number sizes the descriptors, and only the device knows it
        WRAP_TRY(cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, counts, base, n + 1, st));
        *launches += 2;   // (DeviceScan: an initialisation and a scan kernel)
        uint64_t total = 0;
        WRAP_TRY(cudaMemcpyAsync(&total, base + n, sizeof(total), cudaMemcpyDeviceToHost, st));
        WRAP_TRY(cudaStreamSynchronize(st));
        m = n + total;
        if (m > 0xFFFFFFF0ull) return cudaErrorInvalidValue;   // a core launch counts its streams in 32 bits
        const uint64_t k = total;
        WRAP_TRY(scr.slots.reserve(slot_bytes(m) + slot_bytes(n) + slot_bytes(k) + ((k * sizeof(WrapSub) + 15) & ~15ull)));
        Carve cs{static_cast<uint8_t*>(scr.slots.p)};
        A = take_slots(cs, m);
        B = take_slots(cs, n);   // LZ11 over the stream slots: A's offsets
        R = take_slots(cs, k);   // the redo over the chunk slots: A's offsets, its own lengths, capacities and results
        chunk_subs = cs.take<WrapSub>(k);
        A.key = B.key = R.key = nullptr;
        B.src_off = A.src_off;
        B.dst_off = A.dst_off;
        R.src_off = A.src_off + n;
        R.dst_off = A.dst_off + n;
        wrap_chunk_fill_kernel<<<grid, 128, 0, st>>>(d_src_base, d_src_off, d_src_len, d_dst_off, d_dst_cap, N, plans, subs, base, A, B,
                                                     chunk_subs);
        WRAP_TRY(cudaGetLastError());
        ++*launches;
    }

    const uint8_t* src = d_src_base;
    if (format == AURORA_FMT_LZ00) {
        // the keystream is lifted from a device copy of the source: the caller's bytes stay as they are
        WRAP_TRY(scr.src.reserve(src_total + 16));
        WRAP_TRY(cudaMemcpyAsync(scr.src.p, d_src_base, src_total, cudaMemcpyDeviceToDevice, st));
        WRAP_TRY(launch_lcg_xor(static_cast<uint8_t*>(scr.src.p), A.src_off, A.src_len, nullptr, A.key, 0, N, st));
        ++*launches;
        src = static_cast<const uint8_t*>(scr.src.p);
    }

    WRAP_TRY(cudaMemsetAsync(ticket, 0, 64, st));
    auto run = [&](int core, bool headerless, const WrapSlots& S, uint64_t count, unsigned int* t) -> cudaError_t {
        DecodeParams P{};
        fill_decode_params(P, core, &o);   // (the LzProperties of every wrapper format are valid: no override)
        P.headerless = headerless;
        P.src_base = src;
        P.src_limit = (src_total + 15) & ~15ull;
        P.src_off = S.src_off;
        P.src_len = S.src_len;
        P.dst_base = d_dst_base;
        P.dst_off = S.dst_off;
        P.dst_cap = S.dst_cap;
        P.out_len = S.out_len;
        P.consumed = S.consumed;
        P.status = S.status;
        P.order = nullptr;
        P.ticket = t;
        P.n = uint32_t(count);
        ++*launches;
        return launch_decode(P, sm_count, st);
    };
    WRAP_TRY(run(cores.core, cores.headerless, A, m, ticket));
    if (lz77) {
        WRAP_TRY(run(AURORA_FMT_LZ11, false, B, n, ticket + 1));
        wrap_redo_select_kernel<<<grid, 128, 0, st>>>(N, plans, base, A, R);
        WRAP_TRY(cudaGetLastError());
        ++*launches;
        WRAP_TRY(run(AURORA_FMT_LZ10, false, R, m - n, ticket + 2));
    }
    if (format == AURORA_FMT_LEVEL5 || format == AURORA_FMT_ECD) {   // the formats with stored bytes
        wrap_store_kernel<<<(N + 3) / 4, 128, 0, st>>>(d_src_base, d_src_off, d_dst_base, d_dst_off, plans, N);
        WRAP_TRY(cudaGetLastError());
        ++*launches;
    }
    wrap_merge_kernel<<<grid, 128, 0, st>>>(format, N, plans, subs, chunk_subs, base, A, B, cores.core2, d_out_len, d_consumed, d_status);
    WRAP_TRY(cudaGetLastError());
    ++*launches;
    return cudaSuccess;
}

namespace {
inline void put_le32(uint8_t* p, uint32_t v) { p[0] = uint8_t(v); p[1] = uint8_t(v >> 8); p[2] = uint8_t(v >> 16); p[3] = uint8_t(v >> 24); }
inline void put_be32(uint8_t* p, uint32_t v) { p[3] = uint8_t(v); p[2] = uint8_t(v >> 8); p[1] = uint8_t(v >> 16); p[0] = uint8_t(v >> 24); }
}  // namespace

// GetDecompressedSize of the wrapper formats: a header peek
int wrapped_decoded_size(int format, const uint8_t* p, uint64_t len, uint64_t* out_size) {
    *out_size = 0;
    WrapPlan pl{};
    uint64_t at = 0;
    int core = AURORA_FMT_LZ10;
    switch (format) {
        case AURORA_FMT_GCLZ: if (!match_throw(pl, p, len, "GCLZ", 4)) return pl.status; at = 4; break;
        case AURORA_FMT_CXLZ: if (!match_throw(pl, p, len, "CXLZ", 4)) return pl.status; at = 4; break;
        case AURORA_FMT_COMP: if (!match_throw(pl, p, len, "COMP", 4)) return pl.status; at = 4; core = AURORA_FMT_LZ11; break;
        case AURORA_FMT_LZ_3DS: if (!match_throw(pl, p, len, "3DS-LZ\r\n", 8)) return pl.status; at = 8; break;
        case AURORA_FMT_LZ77: {
            if (!match_throw(pl, p, len, "LZ77", 4)) return pl.status;
            if (len < 8) return AURORA_END_OF_STREAM;
            uint32_t v = uint32_t(p[5]) | (uint32_t(p[6]) << 8) | (uint32_t(p[7]) << 16);
            if (v == 0) {
                if (len < 12) return AURORA_END_OF_STREAM;
                v = le32(p + 8);
            }
            *out_size = v;
            return AURORA_OK;
        }
        case AURORA_FMT_LEVEL5:
            if (len < 5) return AURORA_END_OF_STREAM;
            *out_size = p[4] == 0x78 ? le32(p) : le32(p) >> 3;
            return AURORA_OK;
        case AURORA_FMT_SDPC:
            if (!match_throw(pl, p, len, "SDPC", 4)) return pl.status;
            if (len < 8) return AURORA_END_OF_STREAM;
            *out_size = le32(p + 4);
            return AURORA_OK;
        case AURORA_FMT_LZON:
            if (!match_throw(pl, p, len, lzon_magic(), 8)) return pl.status;
            if (len < 12) return AURORA_END_OF_STREAM;
            *out_size = be32(p + 8);
            return AURORA_OK;
        case AURORA_FMT_LEVEL5_LZSS:
            if (!match_throw(pl, p, len, "SSZL", 4)) return pl.status;
            if (len < 16) return AURORA_END_OF_STREAM;
            *out_size = le32(p + 12);
            return AURORA_OK;
        case AURORA_FMT_ECD:   // ECD.cs:43-51: 0 when the compressed size does not fit the stream
            if (!match_throw(pl, p, len, "ECD", 3)) return pl.status;
            if (len < 12) return AURORA_END_OF_STREAM;
            if (uint64_t(be32(p + 8)) + 0x10 > len) return AURORA_OK;
            if (len < 16) return AURORA_END_OF_STREAM;
            *out_size = be32(p + 12);
            return AURORA_OK;
        default: {
            Family f{};
            if (!family_of(format, f)) return AURORA_INVALID_ARGUMENT;
            if (f.magic_len && !match_throw(pl, p, len, f.magic, f.magic_len)) return pl.status;
            if (len < uint64_t(f.size_off) + 4) return AURORA_END_OF_STREAM;
            *out_size = f.size_big ? be32(p + f.size_off) : le32(p + f.size_off);
            return AURORA_OK;
        }
    }
    return core_decoded_size(core, AURORA_ENDIAN_DEFAULT, p + at, len - at, out_size);   // the LZ10 / LZ11 stream behind the identifier
}

// IsMatchStatic of the wrapper formats: identifier (+ a minimum length), then, for GCLZ / CXLZ / COMP, the LZ10 / LZ11
// heuristic on the bytes behind it (GCLZ.cs:30-31, CXLZ.cs:31-32, COMP.cs:30-31, 3DS-LZ.cs:29-30, LZ77.cs:46-47, LZOn.cs:29-30,
// Level5LZSS.cs:29-30; the LZSS family: AKLZ.cs:31-32, LZ01.cs:33-34, FCMP.cs:31-32, IECP.cs:30-31, MDB4.cs:28-29, LZ00.cs:37-38).
// Level5.IsMatch needs zlib and the file name, LZSega / GCZ have no identifier: NOT_SUPPORTED.
int wrapped_is_match_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                           const uint64_t* src_off, const uint64_t* src_len, uint8_t* match) {
    Family f{};
    const bool family = family_of(format, f);
    if (format == AURORA_FMT_LEVEL5 || (family && !f.magic_len)) return AURORA_NOT_SUPPORTED;
    std::vector<size_t> idx;
    std::vector<uint64_t> so, sl;
    for (size_t i = 0; i < n; i++) {
        const uint8_t* p = src_base + src_off[i];
        const uint64_t len = src_len[i];
        auto id = [&](uint64_t min_len, const void* magic, size_t k) { return min_len < len && std::memcmp(p, magic, k) == 0; };
        bool m;
        switch (format) {
            case AURORA_FMT_GCLZ: m = id(0x8, "GCLZ", 4); break;
            case AURORA_FMT_CXLZ: m = id(0x8, "CXLZ", 4); break;
            case AURORA_FMT_COMP: m = id(0x8, "COMP", 4); break;
            case AURORA_FMT_LZ_3DS: m = id(0x10, "3DS-LZ\r\n", 8); break;
            case AURORA_FMT_LZON: m = id(0x10, lzon_magic(), 8); break;
            case AURORA_FMT_LEVEL5_LZSS: m = id(0x10, "SSZL", 4) && (p[4] | p[5] | p[6] | p[7]) == 0; break;
            case AURORA_FMT_LZ77: m = id(0x8, "LZ77", 4) && (p[4] == 0x10 || p[4] == 0x11 || p[4] == 0x24 || p[4] == 0x28 || p[4] == 0x30 || p[4] == 0xF7); break;
            case AURORA_FMT_SDPC: m = id(0x10, "SDPC", 4) && (p[4] | p[5] | p[6] | p[7]) != 0; break;   // SDPC.cs:31-32
            case AURORA_FMT_ECD:   // ECD.cs:37-38: identifier, the compressed size fits the stream, a non-zero decoded size
                m = id(0x10, "ECD", 3) && uint64_t(be32(p + 8)) + 0x10 <= len && be32(p + 12) != 0;
                break;
            default: m = id(format == AURORA_FMT_LZ00 ? 0x40 : 0x10, f.magic, f.magic_len); break;
        }
        match[i] = m ? 1 : 0;
        if (m && (format == AURORA_FMT_GCLZ || format == AURORA_FMT_CXLZ || format == AURORA_FMT_COMP)) {
            idx.push_back(i);
            so.push_back(src_off[i] + 4);
            sl.push_back(len - 4);
        }
    }
    if (!idx.empty()) {
        std::vector<uint8_t> mm(idx.size());
        const int rc = aurora_is_match_batch(ctx, format == AURORA_FMT_COMP ? AURORA_FMT_LZ11 : AURORA_FMT_LZ10, opts, idx.size(),
                                             src_base, so.data(), sl.data(), mm.data());
        if (rc != AURORA_OK) return rc;
        for (size_t k = 0; k < idx.size(); k++) match[idx[k]] = mm[k];
    }
    return AURORA_OK;
}

uint64_t wrapped_encode_bound(int format, uint64_t raw_len, const aurora_codec_opts* opts) {
    switch (format) {
        case AURORA_FMT_GCLZ: case AURORA_FMT_CXLZ: return 4 + aurora_encode_bound(AURORA_FMT_LZ10, raw_len);
        case AURORA_FMT_COMP: return 4 + aurora_encode_bound(AURORA_FMT_LZ11, raw_len);
        case AURORA_FMT_LZ_3DS: return 8 + aurora_encode_bound(AURORA_FMT_LZ10, raw_len);
        case AURORA_FMT_LZ77: {
            const uint64_t chunk = (opts && opts->lz77_chunk_size) ? opts->lz77_chunk_size : 0x1000;
            const uint64_t segs = (raw_len + chunk - 1) / chunk + 1;
            return 8 + 2 * segs + segs * aurora_encode_bound(AURORA_FMT_LZ10, chunk) +
                   std::max(aurora_encode_bound(AURORA_FMT_LZ10, raw_len), aurora_encode_bound(AURORA_FMT_LZ11, raw_len));
        }
        case AURORA_FMT_LEVEL5: return 8 + std::max<uint64_t>(raw_len, aurora_encode_bound(AURORA_FMT_LZ10, raw_len));
        case AURORA_FMT_LZON: return 16 + aurora_encode_bound(AURORA_FMT_LZO, raw_len);
        case AURORA_FMT_SDPC: return 8 + aurora_encode_bound(AURORA_FMT_LZO, raw_len);
        case AURORA_FMT_LEVEL5_LZSS: return 16 + aurora_encode_bound(AURORA_FMT_LZSS, raw_len);
        case AURORA_FMT_ECD: return 16 + std::max<uint64_t>(raw_len, 16 + aurora_encode_bound(AURORA_FMT_LZSS, raw_len));
        default: {
            Family f{};
            return family_of(format, f) ? 64 + aurora_encode_bound(AURORA_FMT_LZSS, raw_len) : 0;
        }
    }
}

// Compress of the wrapper formats: the core encoder writes at the offset the wrapper header leaves free, the header
// bytes are written (or the core's own header is rewritten in place) on the host afterwards.
int wrapped_encode_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                         const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                         const uint64_t* dst_cap, uint64_t* out_len, int32_t* status) {
    aurora_codec_opts o;
    if (opts) o = *opts;
    else aurora_codec_opts_init(&o);
    const bool has_ext = o.struct_size >= sizeof(aurora_codec_opts);
    const uint32_t lz77_type = (has_ext && o.lz77_type) ? o.lz77_type : 0x10;
    const uint64_t chunk = (has_ext && o.lz77_chunk_size) ? o.lz77_chunk_size : 0x1000;
    const uint32_t level5_type = (o.quality == 0) ? 0 : ((has_ext && o.level5_type) ? o.level5_type : 1);

    const uint64_t ecd_plain = (has_ext && o.ecd_plain_size) ? o.ecd_plain_size : 4;   // ECD.PlainSize
    auto ecd_stored = [&](uint64_t len) { return o.quality == 0 || len <= 0x10; };    // ECD.cs:91
    const uint32_t lz00_key = has_ext ? o.lz00_key : 0;

    int core = AURORA_FMT_LZ10;
    uint64_t head = 4;   // bytes in front of the core's output
    switch (format) {
        case AURORA_FMT_GCLZ: case AURORA_FMT_CXLZ: break;
        case AURORA_FMT_COMP: core = AURORA_FMT_LZ11; break;
        case AURORA_FMT_LZ_3DS: head = 8; break;
        case AURORA_FMT_LZ77:
            if (lz77_type == 0x11) core = AURORA_FMT_LZ11;
            else if (lz77_type != 0x10 && lz77_type != 0xF7) {
                for (size_t i = 0; i < n; i++) { status[i] = AURORA_NOT_SUPPORTED; out_len[i] = 0; }
                return AURORA_OK;
            }
            break;
        case AURORA_FMT_LEVEL5:
            if (level5_type > 1) {
                for (size_t i = 0; i < n; i++) { status[i] = AURORA_NOT_SUPPORTED; out_len[i] = 0; }
                return AURORA_OK;
            }
            head = 0;   // the LZ10 header is rewritten in place
            break;
        case AURORA_FMT_LZON: core = AURORA_FMT_LZO; head = 16; break;
        case AURORA_FMT_SDPC: core = AURORA_FMT_LZO; head = 8; break;
        case AURORA_FMT_LEVEL5_LZSS:
            core = AURORA_FMT_LZSS;
            head = 0;   // the 16-byte LZSS header is rewritten in place
            aurora_lz_props_window(&o.lzss, 0x1000, 0xF + 3, 3, 0xFEE, 1);
            break;
        case AURORA_FMT_ECD:
            // header (16) + plain bytes, then the body: the LZSS core's own 16-byte header lands on [plain, plain + 16)
            core = AURORA_FMT_LZSS;
            head = ecd_plain;
            aurora_lz_props_window(&o.lzss, 0x400, 0x42, 3, 0x3BE, 1);
            break;
        default: {
            Family f{};
            if (!family_of(format, f)) return AURORA_INVALID_ARGUMENT;
            // The LZSS core writes its own 16-byte header in front of the body.  It is placed so that the body starts right
            // behind the family's header (header >= 16 bytes), or the body is moved down afterwards (header < 16 bytes).
            core = AURORA_FMT_LZSS;
            const uint64_t hlen = f.read_len + f.skip_len;
            head = hlen >= 16 ? hlen - 16 : 0;
            family_props(f, &o.lzss);
            break;
        }
    }

    // sub-buffers: one per stream, or one per chunk for LZ77 ChunkLZ10 with more than one chunk
    struct Piece { size_t stream; uint64_t soff, slen, doff; };
    std::vector<Piece> pieces;
    std::vector<uint64_t> table_at(n, 0);   // chunked: offset of the u16 table inside the stream's slot
    for (size_t i = 0; i < n; i++) {
        status[i] = AURORA_OK;
        out_len[i] = 0;
        const uint64_t len = src_len[i];
        if (format == AURORA_FMT_LEVEL5 && level5_type == 0) continue;   // stored on the host below
        if (format == AURORA_FMT_ECD) {
            if (ecd_stored(len)) continue;                                   // stored on the host below
            if (ecd_plain > len) { status[i] = AURORA_INVALID_ARGUMENT; continue; }   // source.Slice(0, plainSize)
            if (dst_cap[i] < head) { status[i] = AURORA_DST_TOO_SMALL; continue; }
            pieces.push_back(Piece{i, ecd_plain, len - ecd_plain, head});
            continue;
        }
        if (format == AURORA_FMT_LZ77 && lz77_type == 0xF7 && chunk < len) {
            const uint64_t segs = (len + chunk - 1) / chunk;
            const uint64_t body = 8 + 2 * segs;
            const uint64_t per = aurora_encode_bound(AURORA_FMT_LZ10, chunk);
            if (body + segs * per > dst_cap[i]) { status[i] = AURORA_DST_TOO_SMALL; continue; }
            table_at[i] = 8;
            for (uint64_t k = 0; k < segs; k++)   // encode every chunk into its own worst-case slot, compact afterwards
                pieces.push_back(Piece{i, k * chunk, std::min(chunk, len - k * chunk), body + k * per});
        } else {
            if (dst_cap[i] < head) { status[i] = AURORA_DST_TOO_SMALL; continue; }
            pieces.push_back(Piece{i, 0, len, head});
        }
    }
    const size_t m = pieces.size();
    std::vector<uint64_t> so(m), sl(m), dof(m), dc(m), ol(m);
    std::vector<int32_t> st(m);
    for (size_t j = 0; j < m; j++) {
        const Piece& pc = pieces[j];
        so[j] = src_off[pc.stream] + pc.soff;
        sl[j] = pc.slen;
        dof[j] = dst_off[pc.stream] + pc.doff;
        dc[j] = table_at[pc.stream] ? aurora_encode_bound(AURORA_FMT_LZ10, chunk) : dst_cap[pc.stream] - pc.doff;
    }
    if (m) {
        std::vector<uint32_t> keys;
        if (format == AURORA_FMT_LZ00) keys.assign(m, lz00_key);   // the body goes under the keystream on the device
        const int rc = encode_core_batch(ctx, core, &o, m, src_base, so.data(), sl.data(), dst_base, dof.data(), dc.data(), ol.data(),
                                         st.data(), keys.empty() ? nullptr : keys.data(), 16);
        if (rc != AURORA_OK) return rc;
    }

    // headers
    size_t j = 0;
    for (size_t i = 0; i < n; i++) {
        uint8_t* d = dst_base + dst_off[i];
        const uint64_t len = src_len[i];
        if (format == AURORA_FMT_LEVEL5 && level5_type == 0) {
            if (dst_cap[i] < 4 + len) { status[i] = AURORA_DST_TOO_SMALL; continue; }
            put_le32(d, uint32_t(len) << 3);
            std::memcpy(d + 4, src_base + src_off[i], size_t(len));
            out_len[i] = 4 + len;
            continue;
        }
        if (format == AURORA_FMT_ECD) {   // ECD.cs:88-121
            auto store = [&]() {
                if (dst_cap[i] < 16 + len) { status[i] = AURORA_DST_TOO_SMALL; return; }
                std::memcpy(d, "ECD", 4);   // identifier + flag 0
                put_be32(d + 4, 0);
                put_be32(d + 8, uint32_t(len));
                put_be32(d + 12, uint32_t(len));
                std::memcpy(d + 16, src_base + src_off[i], size_t(len));
                status[i] = AURORA_OK;
                out_len[i] = 16 + len;
            };
            if (ecd_stored(len)) { store(); continue; }
            if (status[i] != AURORA_OK) continue;
            const uint64_t clen = ol[j];
            const int cst = st[j];
            j++;
            // compressed size = plain bytes + body; not smaller than the input (or no room for it): stored instead
            if (cst == AURORA_DST_TOO_SMALL || (cst == AURORA_OK && ecd_plain + (clen - 16) >= len)) { store(); continue; }
            if (cst != AURORA_OK) { status[i] = cst; continue; }
            std::memmove(d + 16, src_base + src_off[i], size_t(ecd_plain));   // overwrites the LZSS core's header
            std::memcpy(d, "ECD\x01", 4);
            put_be32(d + 4, uint32_t(ecd_plain));
            put_be32(d + 8, uint32_t(ecd_plain + clen - 16));
            put_be32(d + 12, uint32_t(len));
            out_len[i] = 16 + ecd_plain + clen - 16;
            continue;
        }
        if (status[i] != AURORA_OK) continue;
        if (table_at[i]) {
            const uint64_t segs = (len + chunk - 1) / chunk;
            const uint64_t body = 8 + 2 * segs;
            std::memcpy(d, "LZ77", 4);
            put_le32(d + 4, 0xF7u | (uint32_t(len) << 8));
            uint64_t end = 0;
            for (uint64_t k = 0; k < segs; k++, j++) {
                if (st[j] != AURORA_OK && status[i] == AURORA_OK) status[i] = st[j];
                if (status[i] != AURORA_OK) continue;
                std::memmove(d + body + end, d + pieces[j].doff, size_t(ol[j]));
                end += ol[j];
                if (end > 0xFFFF) { status[i] = AURORA_INVALID_ARGUMENT; continue; }   // "chunks too large to process"
                d[8 + 2 * k] = uint8_t(end);
                d[8 + 2 * k + 1] = uint8_t(end >> 8);
            }
            if (status[i] == AURORA_OK) out_len[i] = body + end;
            continue;
        }
        const uint64_t clen = ol[j];
        const int cst = st[j];
        j++;
        if (cst != AURORA_OK) { status[i] = cst; continue; }
        switch (format) {
            case AURORA_FMT_GCLZ: std::memcpy(d, "GCLZ", 4); break;
            case AURORA_FMT_CXLZ: std::memcpy(d, "CXLZ", 4); break;
            case AURORA_FMT_COMP: std::memcpy(d, "COMP", 4); break;
            case AURORA_FMT_LZ77: std::memcpy(d, "LZ77", 4); break;
            case AURORA_FMT_LZ_3DS: std::memcpy(d, "3DS-LZ\r\n", 8); break;
            case AURORA_FMT_SDPC:
                std::memcpy(d, "SDPC", 4);
                put_le32(d + 4, uint32_t(len));
                break;
            case AURORA_FMT_LZON:
                std::memcpy(d, lzon_magic(), 8);
                put_be32(d + 8, uint32_t(len));
                put_be32(d + 12, uint32_t(clen));
                break;
            case AURORA_FMT_LEVEL5: {
                // LZ10.Compress wrote 0x10 + u24 (or 0x10 00 00 00 + u32): CompressHeaderless is the same bytes without it
                const uint64_t h = (d[1] | d[2] | d[3]) == 0 ? 8 : 4;
                if (h == 8) std::memmove(d + 4, d + 8, size_t(clen - 8));
                put_le32(d, 1u | (uint32_t(len) << 3));
                out_len[i] = clen - h + 4;
                continue;
            }
            case AURORA_FMT_LEVEL5_LZSS:
                std::memcpy(d, "SSZL", 4);
                put_le32(d + 4, 0);
                put_le32(d + 8, uint32_t(clen - 16));
                put_le32(d + 12, uint32_t(len));
                break;
            default: {
                Family f{};
                family_of(format, f);
                const uint64_t hlen = f.read_len + f.skip_len, blen = clen - 16;   // body bytes (CompressHeaderless)
                if (hlen < 16) std::memmove(d + hlen, d + 16, size_t(blen));
                std::memset(d, 0, size_t(hlen));
                if (f.magic_len) std::memcpy(d, f.magic, f.magic_len);
                switch (format) {
                    case AURORA_FMT_AKLZ: put_be32(d + 12, uint32_t(len)); break;
                    case AURORA_FMT_LZ01: put_le32(d + 4, uint32_t(16 + blen)); put_le32(d + 8, uint32_t(len)); break;   // LZ01.cs:80-81: the whole file
                    case AURORA_FMT_FCMP: put_le32(d + 4, uint32_t(len)); put_le32(d + 8, 305397760u); break;
                    case AURORA_FMT_IECP: put_le32(d + 4, uint32_t(len)); break;
                    case AURORA_FMT_MDB4: put_le32(d + 4, uint32_t(len) + 1); put_le32(d + 8, uint32_t(len)); put_le32(d + 12, uint32_t(32 + blen - 0x10)); break;   // MDB4.cs:78
                    case AURORA_FMT_LZSEGA: put_le32(d, uint32_t(blen)); put_le32(d + 4, uint32_t(len)); break;
                    case AURORA_FMT_GCZ: put_le32(d, uint32_t(len)); break;
                    case AURORA_FMT_LZ00:   // LZ00.cs:86-110
                        put_le32(d + 4, uint32_t(64 + blen));
                        std::memcpy(d + 16, "Temp.dat", 8);   // LZ00.Name default, zero padded to 32 bytes
                        put_le32(d + 48, uint32_t(len));
                        put_le32(d + 52, lz00_key);
                        break;
                }
                out_len[i] = hlen + blen;
                continue;
            }
        }
        out_len[i] = head + clen;
    }
    return AURORA_OK;
}

}  // namespace aurora
