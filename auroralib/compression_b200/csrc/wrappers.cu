// wrappers.cu — the wrapper formats of AuroraLib.Compression.Nintendo (SURVEY.md 8f item 2): a header around one of the
// cores the kernels decode.  Every stream becomes one (ChunkLZ10: several independent) sub-stream of a core batch that runs
// on the device exactly like a direct call.  The header rule (wrap_resolve, wrap_chunk), the merge of the core results
// (wrap_merge) and the ChunkLZ10 redo selection (wrap_redo_chunk) are written once, above the "// ---- kernel" line, and are
// __host__ __device__: aurora_decode_batch resolves the headers on the host, aurora_decode_batch_device in
// wrap_resolve_kernel, one thread per stream.  The encode rules (wrap_encode_plan: a stream's core pieces; wrap_encode_finish:
// its status, header and the copies / moves around the core output) sit there too: aurora_encode_batch applies them on the
// host, aurora_encode_batch_device in wrap_enc_plan_kernel and wrap_enc_finish_kernel.
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

// LZSS-property family: identifier (nullptr: none), header bytes that are READ (a short stream is END_OF_STREAM), bytes skipped by a seek
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
        case AURORA_FMT_LZSEGA: f = Family{format, nullptr, 0, 8, 0, 4, false, false}; return true;
        case AURORA_FMT_GCZ: f = Family{format, nullptr, 0, 4, 0, 0, false, true}; return true;
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

// ---- encode rules: the core encoder writes at an offset the wrapper header leaves free, then the header is written (or the
// core's own header is rewritten in place).  aurora_encode_batch applies them on the host, aurora_encode_batch_device in
// wrap_enc_plan_kernel (one thread per stream) and wrap_enc_finish_kernel (one warp per stream).

__host__ __device__ inline void put_le32(uint8_t* p, uint32_t v) { p[0] = uint8_t(v); p[1] = uint8_t(v >> 8); p[2] = uint8_t(v >> 16); p[3] = uint8_t(v >> 24); }
__host__ __device__ inline void put_be32(uint8_t* p, uint32_t v) { p[3] = uint8_t(v); p[2] = uint8_t(v >> 8); p[1] = uint8_t(v >> 16); p[0] = uint8_t(v >> 24); }
__host__ __device__ inline void put_bytes(uint8_t* p, const char* s, uint64_t k) {
    for (uint64_t j = 0; j < k; j++) p[j] = uint8_t(s[j]);
}
// identifiers as little-endian words, folded at compile time (a string literal in device code would be one more global object)
__host__ __device__ constexpr uint32_t le_word(const char* s) {
    return uint32_t(uint8_t(s[0])) | (uint32_t(uint8_t(s[1])) << 8) | (uint32_t(uint8_t(s[2])) << 16) | (uint32_t(uint8_t(s[3])) << 24);
}
constexpr uint32_t kIdGCLZ = le_word("GCLZ"), kIdCXLZ = le_word("CXLZ"), kIdCOMP = le_word("COMP"), kId3DS0 = le_word("3DS-"),
                   kId3DS1 = le_word("LZ\r\n"), kIdLZ77 = le_word("LZ77"), kIdSDPC = le_word("SDPC"), kIdSSZL = le_word("SSZL"),
                   kIdECD = le_word("ECD\0"), kIdTemp0 = le_word("Temp"), kIdTemp1 = le_word(".dat");

// the options of a wrapped encode, resolved once per batch
struct WrapEnc {
    int format;
    int status;            // OK, or the status of every stream: NOT_SUPPORTED for an LZ77 / Level5 sub-type without an encoder
    int core;              // AURORA_FMT_LZ10 / LZ11 / LZSS / LZO
    uint64_t head;         // bytes in front of the core's output
    uint32_t lz77_type, level5_type, lz00_key;
    uint64_t chunk;        // LZ77.ChunkSize
    uint64_t ecd_plain;    // ECD.PlainSize
    bool quality0;         // quality 0: Level5 and ECD store
};

// false: not a wrapper format.  The extension fields of the option block count only when the caller's block has them.
inline bool wrap_encode_opts(int format, const aurora_codec_opts& o, WrapEnc& e) {
    const bool has_ext = o.struct_size >= sizeof(aurora_codec_opts);
    e.format = format;
    e.status = AURORA_OK;
    e.core = AURORA_FMT_LZ10;
    e.head = 4;
    e.lz77_type = (has_ext && o.lz77_type) ? o.lz77_type : 0x10;
    e.chunk = (has_ext && o.lz77_chunk_size) ? o.lz77_chunk_size : 0x1000;
    e.level5_type = (o.quality == 0) ? 0 : ((has_ext && o.level5_type) ? o.level5_type : 1);
    e.lz00_key = has_ext ? o.lz00_key : 0;
    e.ecd_plain = (has_ext && o.ecd_plain_size) ? o.ecd_plain_size : 4;   // ECD.PlainSize
    e.quality0 = o.quality == 0;
    switch (format) {
        case AURORA_FMT_GCLZ: case AURORA_FMT_CXLZ: break;
        case AURORA_FMT_COMP: e.core = AURORA_FMT_LZ11; break;
        case AURORA_FMT_LZ_3DS: e.head = 8; break;
        case AURORA_FMT_LZ77:
            if (e.lz77_type == 0x11) e.core = AURORA_FMT_LZ11;
            else if (e.lz77_type != 0x10 && e.lz77_type != 0xF7) e.status = AURORA_NOT_SUPPORTED;
            break;
        case AURORA_FMT_LEVEL5:
            if (e.level5_type > 1) e.status = AURORA_NOT_SUPPORTED;
            e.head = 0;   // the LZ10 header is rewritten in place
            break;
        case AURORA_FMT_LZON: e.core = AURORA_FMT_LZO; e.head = 16; break;
        case AURORA_FMT_SDPC: e.core = AURORA_FMT_LZO; e.head = 8; break;
        case AURORA_FMT_LEVEL5_LZSS: e.core = AURORA_FMT_LZSS; e.head = 0; break;   // the 16-byte LZSS header is rewritten in place
        case AURORA_FMT_ECD:
            // header (16) + plain bytes, then the body: the LZSS core's own 16-byte header lands on [plain, plain + 16)
            e.core = AURORA_FMT_LZSS;
            e.head = e.ecd_plain;
            break;
        default: {
            Family f{};
            if (!family_of(format, f)) return false;
            // The LZSS core writes its own 16-byte header in front of the body.  It is placed so that the body starts right
            // behind the family's header (header >= 16 bytes), or the body is moved down afterwards (header < 16 bytes).
            e.core = AURORA_FMT_LZSS;
            const uint64_t hlen = f.read_len + f.skip_len;
            e.head = hlen >= 16 ? hlen - 16 : 0;
            break;
        }
    }
    return true;
}

// The plan of one stream of `len` raw bytes with a destination of `cap` bytes: its up-front status (a stream that is not OK
// runs no core piece and reports out_len 0), whether it is stored, and how many core pieces it has (wrap_encode_piece)
struct WrapEncPlan {
    int status;
    bool stored;    // Level5 OnlySave / ECD stored: no core piece, the finish rule copies the source
    bool chunked;   // ChunkLZ10 with more than one chunk: the u16 end-offset table at 8, the chunks behind it
    uint64_t len, cap;
    uint64_t pieces;   // 0, 1, or the chunk count
};
// one core piece: source bytes [soff, soff + slen) of the stream, encoded to [doff, doff + dcap) of its destination window
struct WrapEncPiece {
    uint64_t soff, slen, doff, dcap;
};

// ChunkLZ10: every chunk is encoded into its own worst-case slot and compacted afterwards
__host__ __device__ inline uint64_t wrap_chunk_slot(const WrapEnc& e) { return core_encode_bound(AURORA_FMT_LZ10, e.chunk); }

__host__ __device__ inline WrapEncPlan wrap_encode_plan(const WrapEnc& e, uint64_t len, uint64_t cap) {
    WrapEncPlan pl{e.status, false, false, len, cap, 0};
    if (e.status != AURORA_OK) return pl;
    if (e.format == AURORA_FMT_LEVEL5 && e.level5_type == 0) {
        pl.stored = true;
        if (cap < 4 + len) pl.status = AURORA_DST_TOO_SMALL;
        return pl;
    }
    if (e.format == AURORA_FMT_ECD) {
        if (e.quality0 || len <= 0x10) {   // ECD.cs:91
            pl.stored = true;
            if (cap < 16 + len) pl.status = AURORA_DST_TOO_SMALL;
            return pl;
        }
        if (e.ecd_plain > len) {   // source.Slice(0, plainSize)
            pl.status = AURORA_INVALID_ARGUMENT;
            return pl;
        }
    }
    if (e.format == AURORA_FMT_LZ77 && e.lz77_type == 0xF7 && e.chunk < len) {
        const uint64_t segs = (len + e.chunk - 1) / e.chunk;
        if (8 + 2 * segs + segs * wrap_chunk_slot(e) > cap) {
            pl.status = AURORA_DST_TOO_SMALL;
            return pl;
        }
        pl.chunked = true;
        pl.pieces = segs;
        return pl;
    }
    if (cap < e.head) {
        pl.status = AURORA_DST_TOO_SMALL;
        return pl;
    }
    pl.pieces = 1;
    return pl;
}

// piece k < pl.pieces
__host__ __device__ inline WrapEncPiece wrap_encode_piece(const WrapEnc& e, const WrapEncPlan& pl, uint64_t k) {
    if (pl.chunked) {
        const uint64_t per = wrap_chunk_slot(e), at = k * e.chunk;
        return WrapEncPiece{at, umin(e.chunk, pl.len - at), 8 + 2 * pl.pieces + k * per, per};
    }
    const uint64_t skip = e.format == AURORA_FMT_ECD ? e.ecd_plain : 0;   // ECD's plain prefix is stored, not encoded
    return WrapEncPiece{skip, pl.len - skip, e.head, pl.cap - e.head};
}

// The finish rule: the stream's status and out_len from its plan and its pieces' results (r_out / r_st[k], k < pl.pieces),
// and what is left to write, in this order: a copy from the source, a downward move inside the window, the ChunkLZ10
// compaction (wrap_encode_chunk_move), then the header bytes (wrap_encode_header).
struct WrapEncFin {
    int status;
    uint64_t out_len;
    bool stored;                             // the stored form (Level5 OnlySave; ECD stored, also as ECD's fall-back)
    uint64_t clen;                           // the core's output length
    uint64_t head_len;                       // header bytes at the start of the window
    uint64_t copy_dst, copy_src, copy_len;   // source bytes [copy_src, copy_src + copy_len) to window offset copy_dst
    uint64_t move_dst, move_src, move_len;   // move_dst < move_src: the ranges may overlap
    uint64_t chunks;                         // ChunkLZ10: chunks 0 .. chunks-1 are compacted, in ascending order
};

__host__ __device__ inline WrapEncFin wrap_encode_finish(const WrapEnc& e, const WrapEncPlan& pl, const uint64_t* r_out, const int32_t* r_st) {
    WrapEncFin f{pl.status, 0, false, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (pl.status != AURORA_OK) return f;
    const uint64_t len = pl.len;
    auto store = [&](uint64_t h) {
        if (pl.cap < h + len) {
            f.status = AURORA_DST_TOO_SMALL;
            return;
        }
        f.stored = true;
        f.head_len = f.copy_dst = h;
        f.copy_len = len;
        f.out_len = h + len;
    };
    if (pl.stored) {
        store(e.format == AURORA_FMT_LEVEL5 ? 4 : 16);
        return f;
    }
    if (pl.chunked) {
        // the header is written whatever the chunks give; the first failing chunk ends the compaction
        f.head_len = 8;
        uint64_t end = 0;
        for (uint64_t k = 0; k < pl.pieces; k++) {
            if (r_st[k] != AURORA_OK) {
                f.status = r_st[k];
                break;
            }
            f.chunks = k + 1;
            end += r_out[k];
            if (end > 0xFFFF) {   // "chunks too large to process"
                f.status = AURORA_INVALID_ARGUMENT;
                break;
            }
        }
        if (f.status == AURORA_OK) f.out_len = 8 + 2 * pl.pieces + end;
        return f;
    }
    const uint64_t clen = r_out[0];
    const int cst = r_st[0];
    f.clen = clen;
    if (e.format == AURORA_FMT_ECD) {   // ECD.cs:88-121
        // compressed size = plain bytes + body; not smaller than the input (or no room for it): stored instead
        if (cst == AURORA_DST_TOO_SMALL || (cst == AURORA_OK && e.ecd_plain + (clen - 16) >= len)) {
            store(16);
            return f;
        }
        if (cst != AURORA_OK) {
            f.status = cst;
            return f;
        }
        f.copy_dst = 16;   // over the LZSS core's header
        f.copy_len = e.ecd_plain;
        f.head_len = 16;
        f.out_len = e.ecd_plain + clen;
        return f;
    }
    if (cst != AURORA_OK) {
        f.status = cst;
        return f;
    }
    f.head_len = e.head;
    f.out_len = e.head + clen;
    if (e.format == AURORA_FMT_LEVEL5) {
        // LZ10.Compress wrote 0x10 + u24 (or, above 0xFFFFFF bytes, 0x10 00 00 00 + u32): CompressHeaderless is the same bytes
        // without it
        const uint64_t h = len > 0xFFFFFF ? 8 : 4;
        if (h == 8) {
            f.move_dst = 4;
            f.move_src = 8;
            f.move_len = clen - 8;
        }
        f.head_len = 4;
        f.out_len = clen - h + 4;
    } else if (e.format == AURORA_FMT_LEVEL5_LZSS) {
        f.head_len = 16;
    } else {
        Family fam{};
        if (family_of(e.format, fam)) {
            const uint64_t hlen = fam.read_len + fam.skip_len;   // the body (CompressHeaderless) goes right behind the header
            if (hlen < 16) {
                f.move_dst = hlen;
                f.move_src = 16;
                f.move_len = clen - 16;
            }
            f.head_len = hlen;
            f.out_len = hlen + clen - 16;
        }
    }
    return f;
}

// ChunkLZ10 compaction step k (k < f.chunks, in ascending order): chunk k moves from its slot to behind the chunks in front of
// it (`end` bytes, updated).  Its destination may overlap earlier chunks' slots, never a later one's: a slot holds at most
// wrap_chunk_slot bytes.  The chunk's u16 end offset goes to 8 + 2k (wrap_encode_table).
struct WrapMove {
    uint64_t dst, src, len;
};
__host__ __device__ inline WrapMove wrap_encode_chunk_move(const WrapEnc& e, const WrapEncPlan& pl, uint64_t k, uint64_t ol, uint64_t& end) {
    const WrapMove m{8 + 2 * pl.pieces + end, wrap_encode_piece(e, pl, k).doff, ol};
    end += ol;
    return m;
}
__host__ __device__ inline void wrap_encode_table(uint8_t* d, uint64_t k, uint64_t end) {
    if (end > 0xFFFF) return;
    d[8 + 2 * k] = uint8_t(end);
    d[8 + 2 * k + 1] = uint8_t(end >> 8);
}

// the f.head_len header bytes at d
__host__ __device__ inline void wrap_encode_header(const WrapEnc& e, const WrapEncPlan& pl, const WrapEncFin& f, uint8_t* d) {
    if (!f.head_len) return;
    const uint32_t len = uint32_t(pl.len);
    const uint64_t clen = f.clen;
    switch (e.format) {
        case AURORA_FMT_GCLZ: put_le32(d, kIdGCLZ); break;
        case AURORA_FMT_CXLZ: put_le32(d, kIdCXLZ); break;
        case AURORA_FMT_COMP: put_le32(d, kIdCOMP); break;
        case AURORA_FMT_LZ_3DS:
            put_le32(d, kId3DS0);
            put_le32(d + 4, kId3DS1);
            break;
        case AURORA_FMT_LZ77:
            put_le32(d, kIdLZ77);
            if (pl.chunked) put_le32(d + 4, 0xF7u | (len << 8));
            break;
        case AURORA_FMT_SDPC:
            put_le32(d, kIdSDPC);
            put_le32(d + 4, len);
            break;
        case AURORA_FMT_LZON:
            put_bytes(d, lzon_magic(), 8);
            put_be32(d + 8, len);
            put_be32(d + 12, uint32_t(clen));
            break;
        case AURORA_FMT_LEVEL5: put_le32(d, f.stored ? len << 3 : 1u | (len << 3)); break;
        case AURORA_FMT_LEVEL5_LZSS:
            put_le32(d, kIdSSZL);
            put_le32(d + 4, 0);
            put_le32(d + 8, uint32_t(clen - 16));
            put_le32(d + 12, len);
            break;
        case AURORA_FMT_ECD:
            put_le32(d, f.stored ? kIdECD : kIdECD | (1u << 24));   // identifier + flag
            put_be32(d + 4, f.stored ? 0u : uint32_t(e.ecd_plain));
            put_be32(d + 8, f.stored ? len : uint32_t(e.ecd_plain + clen - 16));
            put_be32(d + 12, len);
            break;
        default: {
            Family fam{};
            family_of(e.format, fam);
            const uint32_t blen = uint32_t(clen - 16);   // body bytes (CompressHeaderless)
            for (uint64_t j = 0; j < f.head_len; j++) d[j] = 0;
            put_bytes(d, fam.magic, fam.magic_len);
            switch (e.format) {
                case AURORA_FMT_AKLZ: put_be32(d + 12, len); break;
                case AURORA_FMT_LZ01: put_le32(d + 4, 16 + blen); put_le32(d + 8, len); break;   // LZ01.cs:80-81: the whole file
                case AURORA_FMT_FCMP: put_le32(d + 4, len); put_le32(d + 8, 305397760u); break;
                case AURORA_FMT_IECP: put_le32(d + 4, len); break;
                case AURORA_FMT_MDB4: put_le32(d + 4, len + 1); put_le32(d + 8, len); put_le32(d + 12, 32 + blen - 0x10); break;   // MDB4.cs:78
                case AURORA_FMT_LZSEGA: put_le32(d, blen); put_le32(d + 4, len); break;
                case AURORA_FMT_GCZ: put_le32(d, len); break;
                case AURORA_FMT_LZ00:   // LZ00.cs:86-110
                    put_le32(d + 4, 64 + blen);
                    put_le32(d + 16, kIdTemp0);   // LZ00.Name default "Temp.dat", zero padded to 32 bytes
                    put_le32(d + 20, kIdTemp1);
                    put_le32(d + 48, len);
                    put_le32(d + 52, e.lz00_key);
                    break;
            }
            break;
        }
    }
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

// LZ00 decode: the size of every body's 16-byte aligned slot in the keystream-free copy, for the scan (entry n is 0, so the
// scan's entry n is the total)
__global__ void wrap_slot_bytes_kernel(const uint64_t* len, uint32_t n, uint64_t* bytes) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bytes[i] = (len[i] + 15) & ~uint64_t(15);
    if (i == 0) bytes[n] = 0;
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

// ---- encode

// encoder slot j: piece k of a stream at (src_off, dst_off), or (use false) an empty slot — length 0, capacity 0, nothing written
__device__ void put_enc_slot(const WrapSlots& S, uint64_t j, const WrapEnc& e, const WrapEncPlan& pl, uint64_t k, bool use, uint64_t src_off,
                             uint64_t dst_off) {
    const WrapEncPiece pc = use ? wrap_encode_piece(e, pl, k) : WrapEncPiece{0, 0, 0, 0};
    S.src_off[j] = src_off + pc.soff;
    S.src_len[j] = pc.slen;
    S.dst_off[j] = dst_off + pc.doff;
    S.dst_cap[j] = pc.dcap;
    if (S.key) S.key[j] = e.lz00_key;
}

// one thread per stream: the plan and the stream slot (its one piece, else empty); ChunkLZ10 batches write the chunk counts
// instead (entry n stays 0, so the scan's entry n is the total) and leave the slots to wrap_enc_chunk_fill_kernel
__global__ void wrap_enc_plan_kernel(WrapEnc e, const uint64_t* src_off, const uint64_t* src_len, const uint64_t* dst_off, const uint64_t* dst_cap,
                                     uint32_t n, WrapEncPlan* plans, uint64_t* chunks, WrapSlots A) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const WrapEncPlan pl = wrap_encode_plan(e, src_len[i], dst_cap[i]);
    plans[i] = pl;
    if (chunks) {
        chunks[i] = pl.chunked ? pl.pieces : 0;
        if (i == 0) chunks[n] = 0;
    }
    if (A.src_off) put_enc_slot(A, i, e, pl, 0, pl.pieces == 1 && !pl.chunked, src_off[i], dst_off[i]);
}

// ChunkLZ10: stream slot i, then the chunk slots of stream i behind the n stream slots, at n + base[i]
__global__ void wrap_enc_chunk_fill_kernel(WrapEnc e, const uint64_t* src_off, const uint64_t* dst_off, uint32_t n, const WrapEncPlan* plans,
                                           const uint64_t* base, WrapSlots A) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const WrapEncPlan pl = plans[i];
    const uint64_t so = src_off[i], dof = dst_off[i];
    put_enc_slot(A, i, e, pl, 0, pl.pieces == 1 && !pl.chunked, so, dof);
    if (pl.chunked)
        for (uint64_t k = 0; k < pl.pieces; k++) put_enc_slot(A, n + base[i] + k, e, pl, k, true, so, dof);
}

// in-place downward move (d < s, the ranges may overlap), in pieces of 32 x kMoveBytes bytes: every lane loads its bytes of a
// piece before any lane stores them, and the pieces go in ascending order, so no store lands on a byte a later load reads
constexpr int kMoveBytes = 16;
__device__ void warp_move_down(uint8_t* d, const uint8_t* s, uint64_t len, uint32_t lane) {
    for (uint64_t at = 0; at < len; at += 32 * kMoveBytes) {
        uint8_t v[kMoveBytes];
#pragma unroll
        for (int j = 0; j < kMoveBytes; j++) {
            const uint64_t p = at + j * 32 + lane;
            if (p < len) v[j] = s[p];
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < kMoveBytes; j++) {
            const uint64_t p = at + j * 32 + lane;
            if (p < len) d[p] = v[j];
        }
        __syncwarp();
    }
}

// one warp per stream: the finish rule over the pieces' results — the stored copy or ECD's plain prefix, the downward move, the
// ChunkLZ10 compaction with its end-offset table, then the header bytes and the caller's out_len / status
__global__ void wrap_enc_finish_kernel(WrapEnc e, const uint8_t* src, const uint64_t* src_off, uint8_t* dst, const uint64_t* dst_off,
                                       uint32_t n, const WrapEncPlan* plans, const uint64_t* base, WrapSlots A, uint64_t* out_len,
                                       int32_t* status) {
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n) return;
    const WrapEncPlan pl = plans[w];
    const uint64_t j = pl.chunked ? n + base[w] : w;
    const WrapEncFin f = wrap_encode_finish(e, pl, A.out_len + j, A.status + j);
    uint8_t* d = dst + dst_off[w];
    if (f.copy_len) {   // (16-byte accesses when source and destination share their address modulo 16, else 8, 4 or 1 byte)
        uint8_t* cd = d + f.copy_dst;
        const uint8_t* cs = src + src_off[w] + f.copy_src;
        const uintptr_t mis = reinterpret_cast<uintptr_t>(cd) ^ reinterpret_cast<uintptr_t>(cs);
        if ((mis & 15) == 0) warp_copy<uint4>(cd, cs, f.copy_len, lane);
        else if ((mis & 7) == 0) warp_copy<uint2>(cd, cs, f.copy_len, lane);
        else if ((mis & 3) == 0) warp_copy<uint32_t>(cd, cs, f.copy_len, lane);
        else warp_copy<uint8_t>(cd, cs, f.copy_len, lane);
    }
    if (f.move_len) warp_move_down(d + f.move_dst, d + f.move_src, f.move_len, lane);
    uint64_t end = 0;
    for (uint64_t k = 0; k < f.chunks; k++) {
        const WrapMove mv = wrap_encode_chunk_move(e, pl, k, A.out_len[j + k], end);
        if (mv.dst != mv.src) warp_move_down(d + mv.dst, d + mv.src, mv.len, lane);
        if (lane == 0) wrap_encode_table(d, k, end);
    }
    __syncwarp();
    if (lane == 0) {
        wrap_encode_header(e, pl, f, d);
        out_len[w] = f.out_len;
        status[w] = f.status;
    }
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

    const bool lz00 = format == AURORA_FMT_LZ00;

    // per-stream scratch: plans, sub-streams, LZ77's chunk counts (LZ00: its body slots' sizes) and their exclusive scan, the
    // scan's temporary storage
    size_t scan_bytes = 0;
    if (lz77 || lz00)
        WRAP_TRY(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, static_cast<uint64_t*>(nullptr), static_cast<uint64_t*>(nullptr), n + 1, st));
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
    uint64_t src_limit = (src_total + 15) & ~15ull;
    WrapSlots K = A;   // the core launch's slots (LZ00: its bodies are read from their slots in scratch)
    if (lz00) {
        // The keystream is lifted out of place, from the caller's bytes into one 16-byte aligned slot per body: the caller's
        // source stays as it is, and bodies that share source bytes (a file listed twice, windows that overlap) each get
        // their own keystream-free copy.  The slots follow each other in stream order (base[i], the exclusive scan of the
        // aligned body lengths); their total sizes the scratch, and only the device knows the body lengths.
        wrap_slot_bytes_kernel<<<grid, 128, 0, st>>>(A.src_len, N, counts);
        WRAP_TRY(cudaGetLastError());
        ++*launches;
        WRAP_TRY(cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, counts, base, n + 1, st));
        *launches += 2;   // (DeviceScan: an initialisation and a scan kernel)
        uint64_t total = 0;
        WRAP_TRY(cudaMemcpyAsync(&total, base + n, sizeof(total), cudaMemcpyDeviceToHost, st));
        WRAP_TRY(cudaStreamSynchronize(st));
        WRAP_TRY(scr.src.reserve(total + 16));
        WRAP_TRY(launch_lcg_xor(d_src_base, A.src_off, static_cast<uint8_t*>(scr.src.p), base, A.src_len, nullptr, A.key, 0, N, st));
        ++*launches;
        src = static_cast<const uint8_t*>(scr.src.p);
        src_limit = total;
        K.src_off = base;
    }

    WRAP_TRY(cudaMemsetAsync(ticket, 0, 64, st));
    auto run = [&](int core, bool headerless, const WrapSlots& S, uint64_t count, unsigned int* t) -> cudaError_t {
        DecodeParams P{};
        fill_decode_params(P, core, &o);   // (the LzProperties of every wrapper format are valid: no override)
        P.headerless = headerless;
        P.src_base = src;
        P.src_limit = src_limit;
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
    WRAP_TRY(run(cores.core, cores.headerless, K, m, ticket));
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

int wrapped_encode_batch_device(int format, const aurora_codec_opts* opts, size_t n, const uint8_t* d_src_base, uint64_t src_total,
                                const uint64_t* d_src_off, const uint64_t* d_src_len, uint8_t* d_dst_base, const uint64_t* d_dst_off,
                                const uint64_t* d_dst_cap, uint64_t* d_out_len, int32_t* d_status, WrapScratch& scr,
                                DevBuf& enc_scratch, unsigned int* ticket, int sm_count, cudaStream_t st, uint64_t* launches,
                                cudaError_t* err) {
    const aurora_codec_opts o = wrap_core_opts(format, opts);
    WrapEnc e;
    if (!wrap_encode_opts(format, o, e)) return AURORA_INVALID_ARGUMENT;
    EncodeParams P{};
    const int rc = fill_encode_params(P, e.core, &o);   // (the LzProperties of every wrapper format are valid)
    if (rc != AURORA_OK) return rc;
    auto cuda = [&](cudaError_t c) {
        *err = c;
        return c == cudaSuccess ? AURORA_OK : AURORA_CUDA_ERROR;
    };
#define WRAP_ENC_TRY(expr)                                     \
    do {                                                       \
        if (cuda(expr) != AURORA_OK) return AURORA_CUDA_ERROR; \
    } while (0)
    const bool chunked = format == AURORA_FMT_LZ77 && e.lz77_type == 0xF7;
    const uint32_t N = uint32_t(n);
    const unsigned grid = (N + 127) / 128;

    // per-stream scratch: plans, ChunkLZ10's chunk counts and their exclusive scan, the scan's temporary storage
    size_t scan_bytes = 0;
    if (chunked)
        WRAP_ENC_TRY(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, static_cast<uint64_t*>(nullptr), static_cast<uint64_t*>(nullptr), n + 1, st));
    WRAP_ENC_TRY(scr.plans.reserve(((n * sizeof(WrapEncPlan) + 15) & ~15ull) + 2 * (((n + 1) * 8 + 15) & ~15ull) + scan_bytes));
    Carve cp{static_cast<uint8_t*>(scr.plans.p)};
    WrapEncPlan* plans = cp.take<WrapEncPlan>(n);
    uint64_t* counts = cp.take<uint64_t>(n + 1);
    uint64_t* base = cp.take<uint64_t>(n + 1);
    void* scan_tmp = cp.p;

    WrapSlots A{};
    uint64_t m = n;
    if (!chunked) {   // one slot per stream: the plan pass writes them
        WRAP_ENC_TRY(scr.slots.reserve(slot_bytes(n)));
        Carve cs{static_cast<uint8_t*>(scr.slots.p)};
        A = take_slots(cs, n);
        if (format != AURORA_FMT_LZ00) A.key = nullptr;
    }
    wrap_enc_plan_kernel<<<grid, 128, 0, st>>>(e, d_src_off, d_src_len, d_dst_off, d_dst_cap, N, plans, chunked ? counts : nullptr, A);
    WRAP_ENC_TRY(cudaGetLastError());
    ++*launches;
    if (chunked) {
        // the chunk slots follow the n stream slots; their number sizes the descriptors, and only the device knows the lengths
        WRAP_ENC_TRY(cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, counts, base, n + 1, st));
        *launches += 2;   // (DeviceScan: an initialisation and a scan kernel)
        uint64_t total = 0;
        WRAP_ENC_TRY(cudaMemcpyAsync(&total, base + n, sizeof(total), cudaMemcpyDeviceToHost, st));
        WRAP_ENC_TRY(cudaStreamSynchronize(st));
        m = n + total;
        if (m > 0xFFFFFFF0ull) return cuda(cudaErrorInvalidValue);   // a core launch counts its streams in 32 bits
        WRAP_ENC_TRY(scr.slots.reserve(slot_bytes(m)));
        Carve cs{static_cast<uint8_t*>(scr.slots.p)};
        A = take_slots(cs, m);
        A.key = nullptr;
        wrap_enc_chunk_fill_kernel<<<grid, 128, 0, st>>>(e, d_src_off, d_dst_off, N, plans, base, A);
        WRAP_ENC_TRY(cudaGetLastError());
        ++*launches;
    }

    // the core encoder over every slot, as aurora_encode_batch_device runs it (every slot lies inside the src_total bytes)
    P.n = uint32_t(m);
    P.chain_bits = encode_chain_bits(P.chain_bits, src_total);
    const int warps = encode_launch_warps(P, sm_count);
    P.scratch_per_warp = encode_scratch_per_warp(e.core, P.hash_bits, P.chain_bits, 0);   // (no section staging: not MIO0 / Yay0)
    WRAP_ENC_TRY(enc_scratch.reserve(size_t(warps) * P.scratch_per_warp));
    WRAP_ENC_TRY(cudaMemsetAsync(ticket, 0, 64, st));
    P.scratch = static_cast<uint8_t*>(enc_scratch.p);
    P.src_base = d_src_base;
    P.src_limit = src_total;
    P.src_off = A.src_off;
    P.src_len = A.src_len;
    P.dst_base = d_dst_base;
    P.dst_off = A.dst_off;
    P.dst_cap = A.dst_cap;
    P.out_len = A.out_len;
    P.status = A.status;
    P.ticket = ticket;
    WRAP_ENC_TRY(launch_encode(P, warps, st));
    ++*launches;
    if (format == AURORA_FMT_LZ00) {   // the body the encoder just wrote goes under the keystream (bytes [16, out_len) of every piece)
        WRAP_ENC_TRY(launch_lcg_xor(d_dst_base, A.dst_off, d_dst_base, A.dst_off, A.out_len, A.dst_cap, A.key, 16, N, st));
        ++*launches;
    }
    wrap_enc_finish_kernel<<<(N + 3) / 4, 128, 0, st>>>(e, d_src_base, d_src_off, d_dst_base, d_dst_off, N, plans, base, A, d_out_len, d_status);
    WRAP_ENC_TRY(cudaGetLastError());
    ++*launches;
#undef WRAP_ENC_TRY
    return AURORA_OK;
}

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

// Compress of the wrapper formats: the encode rules above, with the core pieces of every stream in one core batch and the
// finish rule's copies, moves and header bytes applied on the host.
int wrapped_encode_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                         const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                         const uint64_t* dst_cap, uint64_t* out_len, int32_t* status) {
    const aurora_codec_opts o = wrap_core_opts(format, opts);
    WrapEnc e;
    if (!wrap_encode_opts(format, o, e)) return AURORA_INVALID_ARGUMENT;
    if (e.status != AURORA_OK) {
        for (size_t i = 0; i < n; i++) { status[i] = e.status; out_len[i] = 0; }
        return AURORA_OK;
    }
    std::vector<WrapEncPlan> plans(n);
    std::vector<size_t> first(n);   // the stream's first piece
    std::vector<uint64_t> so, sl, dof, dc;
    for (size_t i = 0; i < n; i++) {
        plans[i] = wrap_encode_plan(e, src_len[i], dst_cap[i]);
        first[i] = so.size();
        for (uint64_t k = 0; k < plans[i].pieces; k++) {
            const WrapEncPiece pc = wrap_encode_piece(e, plans[i], k);
            so.push_back(src_off[i] + pc.soff);
            sl.push_back(pc.slen);
            dof.push_back(dst_off[i] + pc.doff);
            dc.push_back(pc.dcap);
        }
    }
    const size_t m = so.size();
    std::vector<uint64_t> ol(m + 1, 0);
    std::vector<int32_t> st(m + 1, AURORA_OK);
    if (m) {
        std::vector<uint32_t> keys;
        if (format == AURORA_FMT_LZ00) keys.assign(m, e.lz00_key);   // the body goes under the keystream on the device
        const int rc = encode_core_batch(ctx, e.core, &o, m, src_base, so.data(), sl.data(), dst_base, dof.data(), dc.data(), ol.data(),
                                         st.data(), keys.empty() ? nullptr : keys.data(), 16);
        if (rc != AURORA_OK) return rc;
    }
    for (size_t i = 0; i < n; i++) {
        const WrapEncPlan& pl = plans[i];
        const WrapEncFin f = wrap_encode_finish(e, pl, ol.data() + first[i], st.data() + first[i]);
        uint8_t* d = dst_base + dst_off[i];
        if (f.copy_len) std::memcpy(d + f.copy_dst, src_base + src_off[i] + f.copy_src, size_t(f.copy_len));
        if (f.move_len) std::memmove(d + f.move_dst, d + f.move_src, size_t(f.move_len));
        uint64_t end = 0;
        for (uint64_t k = 0; k < f.chunks; k++) {
            const WrapMove mv = wrap_encode_chunk_move(e, pl, k, ol[first[i] + k], end);
            std::memmove(d + mv.dst, d + mv.src, size_t(mv.len));
            wrap_encode_table(d, k, end);
        }
        wrap_encode_header(e, pl, f, d);
        out_len[i] = f.out_len;
        status[i] = f.status;
    }
    return AURORA_OK;
}

}  // namespace aurora
