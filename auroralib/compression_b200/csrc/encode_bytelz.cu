// encode_bytelz.cu — batched encoders for the byte-tagged formats: LZ4 (block, legacy frame, v1 frame), Snappy (raw
// block and framing format), LZO1X and SEGA PRS.  One raw buffer per warp, exact replay of the reference's match finder
// (finder.cuh), so the output is byte-identical to the reference encoder.
//
// Reference token writers restated (paths under /root/reference/src):
//   LZ4     AuroraLib.Compression/Formats/Common/LZ4.cs:114-160 (Compress), :202-238 (CompressBlockHeaderless),
//           WriteExtension :254-268; LZ4.Frame.cs:176-227 (v1 frame; flags wiped to IsVersion1 :184)
//   Snappy  Formats/Common/Snappy.cs:71-107 (framing, CRC32C masked :252), :130-203 (CompressHeaderless)
//   LZO     Formats/Common/LZO.cs:141-250, WriteExtendedInt :263-271
//   PRS     AuroraLib.Compression.Sega/Sega/PRS.cs:104-159 with FlagWriter.FlushIfNecessary (IO/FlagWriter.cs:132-139)
#include "common.cuh"
#include "finder.cuh"

namespace aurora {

namespace {

// bounded sequential output; lane 0 stores single bytes, runs are copied by the whole warp
struct Out {
    uint8_t* out;
    uint64_t cap, pos;
    bool overflow;
    __device__ __forceinline__ void byte(uint32_t b) {
        if (pos < cap) {
            if (lane_id() == 0) out[pos] = uint8_t(b);
        } else {
            overflow = true;
        }
        pos++;
    }
    __device__ __forceinline__ void at(uint64_t p, uint32_t b) {
        if (p < cap && lane_id() == 0) out[p] = uint8_t(b);
    }
    __device__ __forceinline__ void u16le(uint32_t v) { byte(v & 0xFF); byte((v >> 8) & 0xFF); }
    __device__ __forceinline__ void u24le(uint32_t v) { byte(v & 0xFF); byte((v >> 8) & 0xFF); byte((v >> 16) & 0xFF); }
    __device__ __forceinline__ void u32le(uint32_t v) { u16le(v & 0xFFFF); u16le(v >> 16); }
    __device__ __forceinline__ void patch_u32le(uint64_t p, uint32_t v) {
        for (int i = 0; i < 4; i++) at(p + i, (v >> (8 * i)) & 0xFF);
    }
    __device__ __forceinline__ void patch_u24le(uint64_t p, uint32_t v) {
        for (int i = 0; i < 3; i++) at(p + i, (v >> (8 * i)) & 0xFF);
    }
    __device__ __forceinline__ void copy(const uint8_t* src, uint32_t n) {
        if (pos + n > cap) overflow = true;
        for (uint32_t i = lane_id(); i < n; i += 32)
            if (pos + i < cap) out[pos + i] = src[i];
        pos += n;
    }
};

// ------------------------------------------------------------------------------------------------ LZ4
// LZ4.cs:254-268
__device__ __forceinline__ void lz4_write_ext(Out& o, int length) {
    length -= 0xF;
    if (length >= 0) {
        int b;
        do {
            b = min(length, 0xFF);
            o.byte(uint32_t(b));
            length -= b;
        } while (b == 0xFF);
    }
}

// LZ4.cs:202-238.  A fresh match finder per call.
__device__ int lz4_block_encode(Finder& f, const uint8_t* source, int n, Out& o) {
    if (n < 5) return AURORA_INVALID_ARGUMENT;   // source.Slice(0, Length - 5) throws
    finder_reset(f);
    int sp = 0;
    const int encode_len = n - 5;
    for (;;) {
        const Match m = find_next_best_match(f, source, encode_len);
        int plain = m.offset - sp;
        int token = (plain > 0xF ? 0xF : plain) << 4;
        if (m.length != 0) {
            token |= (m.length - 4 > 0xF ? 0xF : m.length - 4);
        } else {
            plain = n - sp;
            token = (plain > 0xF ? 0xF : plain) << 4;
        }
        o.byte(uint32_t(token));
        lz4_write_ext(o, plain);
        o.copy(source + sp, uint32_t(plain));
        sp += plain;
        if (sp >= n) break;
        o.u16le(uint32_t(m.distance) & 0xFFFF);
        lz4_write_ext(o, m.length - 4);
        sp += m.length;
    }
    return AURORA_OK;
}

// ------------------------------------------------------------------------------------------------ Snappy
__constant__ uint32_t c_crc32c[256];   // reflected CRC-32C table (polynomial 0x82F63B78), filled by the launcher

__device__ uint32_t crc32c_masked(const uint8_t* p, uint32_t n) {
    // every lane walks the bytes (uniform loads, constant-bank table): ~1 % of the chunk's encode time
    uint32_t crc = 0xFFFFFFFFu;
    for (uint32_t i = 0; i < n; i++) crc = c_crc32c[(crc ^ p[i]) & 0xFF] ^ (crc >> 8);
    crc = ~crc;
    return ((crc >> 15) | (crc << 17)) + 0xa282ead8u;   // Snappy.CRCMask (:252)
}

// Snappy.cs:130-203 (the finder is Reset() by the caller between chunks, :86)
__device__ void snappy_block_encode(Finder& f, const uint8_t* source, int n, Out& o) {
    int v = n;
    while (v >= 0x80) {
        o.byte(uint32_t(v | 0x80) & 0xFF);
        v >>= 7;
    }
    o.byte(uint32_t(v));
    int sp = 0;
    for (;;) {
        const Match m = find_next_best_match(f, source, n);
        const int plain = m.offset - sp;
        if (plain > 0) {
            if (plain <= 60) {
                o.byte(uint32_t(plain - 1) << 2);
            } else {
                const uint32_t len = uint32_t(plain - 1);
                if (len <= 0xFF) { o.byte(60 << 2); o.byte(len); }
                else if (len <= 0xFFFF) { o.byte(61 << 2); o.u16le(len); }
                else if (len <= 0xFFFFFF) { o.byte(62 << 2); o.u24le(len); }
                else { o.byte(63 << 2); o.u32le(len); }
            }
            o.copy(source + sp, uint32_t(plain));
            sp += plain;
        }
        if (m.length == 0) return;
        sp += m.length;
        if (m.distance < 2048 && m.length >= 4 && m.length <= 11) {
            o.byte((1u | (uint32_t(m.length - 4) << 2) | (uint32_t(m.distance >> 8) << 5)) & 0xFF);
            o.byte(uint32_t(m.distance) & 0xFF);
        } else {
            o.byte((2u | (uint32_t(m.length - 1) << 2)) & 0xFF);
            o.u16le(uint32_t(m.distance) & 0xFFFF);
        }
    }
}

// ------------------------------------------------------------------------------------------------ LZO
// LZO.cs:263-271
__device__ __forceinline__ void lzo_write_ext(Out& o, int value) {
    while (value > 255) {
        o.byte(0);
        value -= 255;
    }
    o.byte(uint32_t(value));
}

// LZO.cs:141-250
__device__ int lzo_encode(Finder& f, const uint8_t* source, int n, Out& o) {
    if (n < 0x10) {
        o.byte(uint32_t(17 + n));
        o.copy(source, uint32_t(n));
        o.byte(0x11); o.byte(0); o.byte(0);
        return AURORA_OK;
    }
    finder_reset(f);
    int sp = 0;
    Match match = find_next_best_match(f, source, n);
    Match next = find_next_best_match(f, source, n);
    while (sp != n) {
        int plain = match.offset - sp;
        if (plain != 0) {
            if (plain < 4) {
                const int dif = 4 - plain;
                match = Match{match.offset + dif, match.distance, match.length - dif};
                plain = 4;
            }
            if (plain > 18) {
                o.byte(0);
                lzo_write_ext(o, plain - 18);
            } else {
                o.byte(uint32_t(plain - 3));
            }
            if (sp + plain > n) return AURORA_INVALID_ARGUMENT;   // Slice -> ArgumentOutOfRangeException
            o.copy(source + sp, uint32_t(plain));
            sp += plain;
        }
        if (match.length >= 3) {
            sp += match.length;
            plain = next.offset - sp;
            if (plain > 3) plain = 0;
            if (match.length <= 8 && match.distance <= 2048) {
                const uint32_t flag = (uint32_t(plain) | ((uint32_t(match.distance - 1) & 0x7) << 2)) & 0xFF;
                if (match.length <= 4) o.byte((flag | 0x40 | (uint32_t(match.length - 3) << 5)) & 0xFF);
                else o.byte((flag | 0x80 | (uint32_t(match.length - 5) << 5)) & 0xFF);
                o.byte((uint32_t(match.distance - 1) >> 3) & 0xFF);
            } else if (match.distance <= 16384) {
                if (match.length > 33) {
                    o.byte(0x20);
                    lzo_write_ext(o, match.length - 33);
                } else {
                    o.byte((0x20u | uint32_t(match.length - 2)) & 0xFF);
                }
                o.byte((uint32_t(plain) | (uint32_t(match.distance - 1) << 2)) & 0xFF);
                o.byte((uint32_t(match.distance - 1) >> 6) & 0xFF);
            } else {
                const int hflag = 0x4000;
                const int distance = match.distance - hflag;
                const uint32_t flag = (0x10u | (uint32_t(distance & hflag) >> 11)) & 0xFF;
                if (match.length > 9) {
                    o.byte(flag);
                    lzo_write_ext(o, match.length - 9);
                } else {
                    o.byte((flag | uint32_t(match.length - 2)) & 0xFF);
                }
                o.byte((uint32_t(plain) | (uint32_t(distance) << 2)) & 0xFF);
                o.byte((uint32_t(distance) >> 6) & 0xFF);
            }
            if (plain < 0 || sp + plain > n) return AURORA_INVALID_ARGUMENT;
            o.copy(source + sp, uint32_t(plain));
            sp += plain;
        }
        match = next;
        next = find_next_best_match(f, source, n);
    }
    o.byte(0x11); o.byte(0); o.byte(0);
    return AURORA_OK;
}

// ------------------------------------------------------------------------------------------------ PRS
// PRS.cs:104-159.  `Writer` (finder.cuh) reserves the flag byte of a group when its first byte or bit arrives, which is
// the layout FlagWriter produces; the one case that differs — a short match whose 4th control bit completes a flag
// byte, after which FlushIfNecessary emits the distance byte on its own — is written with raw_byte.
__device__ void prs_encode(Finder& f, const uint8_t* source, int n, Writer& w, bool big) {
    finder_reset(f);
    int sp = 0;
    for (;;) {
        const Match m = find_next_best_match(f, source, n);
        int plain = m.offset - sp;
        while (plain != 0) {
            plain--;
            w.byte(source[sp++]);
            w.bit(true);
        }
        if (m.length == 0) break;
        if (m.length == 2 && m.distance > 0x100) continue;
        sp += m.length;
        const int distance = -m.distance;
        const int length = m.length;
        w.bit(false);
        if (distance >= -0x100 && length <= 5) {
            w.bit(false);
            w.bit(((length - 2) >> 1) & 1);
            w.bit((length - 2) & 1);
            if (w.flag_pos < 0) w.raw_byte(uint32_t(distance) & 0xFF);   // FlushIfNecessary: no flag pending
            else w.byte(uint32_t(distance) & 0xFF);
        } else {
            const uint32_t v = (length > 9) ? (uint32_t(distance << 3) & 0xFFFF) : ((uint32_t(distance << 3) | uint32_t(length - 2)) & 0xFFFF);
            if (big) { w.byte(v >> 8); w.byte(v & 0xFF); }
            else { w.byte(v & 0xFF); w.byte(v >> 8); }
            if (length > 9) w.byte(uint32_t(length - 1) & 0xFF);
            w.bit(true);
        }
    }
    w.bit(false);
    w.byte(0);
    w.byte(0);
    w.bit(true);
    w.dispose();
}

__device__ void encode_stream(const EncodeParams& P, uint32_t idx, Finder& f) {
    const uint8_t* src = P.src_base + P.src_off[idx];
    const uint64_t n64 = P.src_len[idx];
    int status = AURORA_OK;
    uint64_t out_len = 0;
    if (n64 > 0x7FFFFFF0ull) {
        status = AURORA_INVALID_ARGUMENT;
    } else {
        const int n = int(n64);
        Out o{P.dst_base + P.dst_off[idx], P.dst_cap[idx], 0, false};
        switch (P.format) {
            case AURORA_FMT_LZ4_BLOCK: status = lz4_block_encode(f, src, n, o); break;
            case AURORA_FMT_LZ4_LEGACY: {   // LZ4.cs:121-134
                o.u32le(0x184C2102u);
                int sp = 0;
                while (sp != n && status == AURORA_OK) {
                    const uint64_t block_start = o.pos;
                    o.u32le(0);
                    const int block_len = min(0x400000 * 2, n - sp);
                    status = lz4_block_encode(f, src + sp, block_len, o);
                    sp += block_len;
                    o.patch_u32le(block_start, uint32_t(o.pos - block_start - 4));
                }
                o.byte(0xFF);
                break;
            }
            case AURORA_FMT_LZ4: {   // LZ4.Frame.cs:176-227
                o.u32le(0x184D2204u);
                const uint32_t bs = P.lz4_block_size;
                o.byte(0x40);
                o.byte(bs == 0x10000 ? 0x40 : bs == 0x40000 ? 0x50 : bs == 0x100000 ? 0x60 : 0x70);
                o.byte(bs == 0x10000 ? 0xC0 : bs == 0x40000 ? 0x77 : bs == 0x100000 ? 0x96 : 0xDF);   // (XXH32(FLG, BD) >> 8) & 0xFF
                int sp = 0;
                while (sp != n && status == AURORA_OK) {
                    const int block_len = min(int(bs), n - sp);
                    const uint64_t hdr = o.pos;
                    o.u32le(0);
                    status = lz4_block_encode(f, src + sp, block_len, o);
                    const uint64_t csize = o.pos - hdr - 4;
                    if (csize >= bs) {   // stored block
                        __syncwarp();   // the attempt's bytes (all lanes copy literals) are overwritten: order the two
                        o.pos = hdr;
                        o.u32le(uint32_t(block_len) | 0x80000000u);
                        o.copy(src + sp, uint32_t(block_len));
                    } else {
                        o.patch_u32le(hdr, uint32_t(csize));
                    }
                    sp += block_len;
                }
                o.u32le(0);
                break;
            }
            case AURORA_FMT_SNAPPY_BLOCK:
                finder_reset(f);
                snappy_block_encode(f, src, n, o);
                break;
            case AURORA_FMT_SNAPPY: {   // Snappy.cs:71-107
                const uint8_t id[10] = {0xff, 0x06, 0x00, 0x00, 0x73, 0x4e, 0x61, 0x50, 0x70, 0x59};
                for (int i = 0; i < 10; i++) o.byte(id[i]);
                int p = 0;
                while (p < n) {
                    const int chunk = min(0x10000, n - p);
                    const uint32_t crc = crc32c_masked(src + p, uint32_t(chunk));
                    const uint64_t hdr = o.pos;
                    o.byte(0);
                    o.u24le(0);
                    o.u32le(crc);
                    finder_reset(f);
                    snappy_block_encode(f, src + p, chunk, o);
                    const uint64_t csize = o.pos - hdr - 8;
                    if (csize >= uint64_t(chunk)) {   // stored chunk
                        __syncwarp();   // (as for LZ4's stored blocks; found by the lane emulation of tests/simt)
                        o.pos = hdr;
                        o.byte(1);
                        o.u24le(uint32_t(chunk + 4));
                        o.u32le(crc);
                        o.copy(src + p, uint32_t(chunk));
                    } else {
                        o.patch_u24le(hdr + 1, uint32_t(csize + 4));
                    }
                    p += chunk;
                }
                break;
            }
            case AURORA_FMT_LZO: status = lzo_encode(f, src, n, o); break;
            case AURORA_FMT_PRS: {
                Writer w;
                w.out = o.out;
                w.cap = o.cap;
                w.pos = 0;
                w.flag_pos = -1;
                w.flag_val = w.bits = 0;
                w.msb_first = P.byte_order != AURORA_ENDIAN_LITTLE;   // FlagWriter(destination, order): bit order = byte order
                w.overflow = false;
                prs_encode(f, src, n, w, P.byte_order != AURORA_ENDIAN_LITTLE);
                o.pos = w.pos;
                o.overflow = w.overflow;
                break;
            }
            default: status = AURORA_NOT_SUPPORTED;
        }
        out_len = o.pos;
        if (status == AURORA_OK && (o.overflow || o.pos > o.cap)) status = AURORA_DST_TOO_SMALL;
    }
    if (lane_id() == 0) {
        P.out_len[idx] = out_len;
        P.status[idx] = status;
    }
    __syncwarp();
}

// ---- kernel
__global__ void __launch_bounds__(kEncWarpsPerBlock * 32) encode_bytelz_kernel(const EncodeParams P) {
    const int warp_global = blockIdx.x * kEncWarpsPerBlock + (threadIdx.x >> 5);
    uint8_t* scratch = P.scratch + size_t(warp_global) * P.scratch_per_warp;
    Finder f;
    finder_setup(f, P, scratch);
    for (;;) {
        uint32_t t = 0;
        if (lane_id() == 0) t = atomicAdd(P.ticket, 1u);
        t = __shfl_sync(kFull, t, 0);
        if (t >= P.n) break;
        encode_stream(P, t, f);
    }
}

}  // namespace

cudaError_t launch_encode_bytelz(const EncodeParams& p, int warps, cudaStream_t st) {
    static bool table_ready[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (!table_ready[dev & 63]) {
        uint32_t t[256];
        for (uint32_t i = 0; i < 256; i++) {
            uint32_t c = i;
            for (int j = 0; j < 8; j++) c = (c & 1) ? (c >> 1) ^ 0x82F63B78u : c >> 1;
            t[i] = c;
        }
        cudaError_t e = cudaMemcpyToSymbol(c_crc32c, t, sizeof(t));
        if (e != cudaSuccess) return e;
        table_ready[dev & 63] = true;
    }
    encode_bytelz_kernel<<<warps / kEncWarpsPerBlock, kEncWarpsPerBlock * 32, 0, st>>>(p);
    return cudaGetLastError();
}

}  // namespace aurora
