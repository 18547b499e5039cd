// encode_lz.cu — batched encoder for the flag-byte LZ77 family (LZ10, LZ11, Yaz0/Yaz1, LZSS, MIO0, Yay0).
// One raw buffer per warp.
//
// Reference semantics restated on the device (paths under /root/reference/src):
//   match finder  AuroraLib.Compression/MatchFinder/LzChainMatchFinder.cs: parameters :108-119, Reset :121-128,
//                 Insert :130-140, FindNextBestMatch :157-212, MatchSearch :214-246, ChainMatches :248-282,
//                 ComputeHash :288-299, GetMatchLength :338-357
//   token writers Nintendo/LZ10.cs:67-80,:113-137; LZ11.cs:65-81,:135-171; Yaz0.cs:82-98 + Yay0.cs:152-184;
//                 Yay0.cs:63-78; MIO0.cs:64-81,:159-184; Formats/Common/LZSS.cs:72-89,:132-160
//   flag packing  AuroraLib.Compression/IO/FlagWriter.cs:70-80 (WriteBit), :111-127 (Flush)
//
// Round-1 design: exact emulation.  The reference's parse is sequential state (head/chain/min tables updated
// as the cursor moves, greedy with one-step lazy lookahead), so each warp replays it for its stream with the
// same hash function and the same table sizes (tables live in a per-warp slice of a global scratch buffer,
// the 4-byte-hash head table is 2 MiB at the default quality 8), which makes the output byte-identical to
// the reference encoder.  The 32 lanes are spent on the parts that are data parallel: the common-prefix
// comparison of every chain candidate (32 bytes per step, ballot for the first mismatch) and the table reset.
// The one-thread-per-window-position search with a shared-memory hash table is the planned replacement
// (DESIGN.md, "what comes next").
// Measured and rejected (round 1): one stream per THREAD with the same tables (32 streams per warp instruction, 32 table
// lookups in flight per warp, epoch-stamped entries instead of per-stream resets).  Byte-identical, but 2.1 GB/s against
// 8.1 GB/s here: the reference-sized tables (2.3 MiB per stream at quality 8) cap the resident streams at ~19 000
// threads = 4 warps per SM, and those warps diverge through the chain walk and the prefix comparison.  A faster exact
// encoder needs compact tables first (e.g. window-sized bucket heads / bucket chains that reproduce head[h] by
// re-hashing the candidates), so that thousands of streams per SM can be resident.
#include "common.cuh"
#include "finder.cuh"

namespace aurora {

namespace {

enum EncKind { E_LZ10 = 0, E_LZ11 = 1, E_YAZ0 = 2, E_LZSS = 3, E_MIO0 = 4, E_YAY0 = 5 };

__device__ __forceinline__ void put_u32(Writer& w, uint32_t v, bool big) {
    for (int i = 0; i < 4; i++) w.raw_byte(big ? (v >> (24 - 8 * i)) & 0xFF : (v >> (8 * i)) & 0xFF);
}

template <int K>
__device__ void encode_stream(const EncodeParams& P, uint32_t idx, Finder& f) {
    const uint8_t* src = P.src_base + P.src_off[idx];
    const uint64_t n64 = P.src_len[idx];
    const int lane = lane_id();
    int status = AURORA_OK;
    uint64_t out_len = 0;
    if (n64 > 0x7FFFFFF0ull) {
        status = AURORA_INVALID_ARGUMENT;
    } else {
        const int n = int(n64);
        finder_reset(f);
        Writer w;
        w.out = P.dst_base + P.dst_off[idx];
        w.cap = P.dst_cap[idx];
        w.pos = 0;
        w.flag_pos = -1;
        w.flag_val = w.bits = 0;
        w.msb_first = K != E_LZSS;
        w.overflow = false;
        const bool big = P.byte_order != AURORA_ENDIAN_LITTLE;   // class default Big

        // split-stream formats assemble three sections; codes and literals are staged behind the flag section
        uint8_t* codes = nullptr;
        uint8_t* lits = nullptr;
        uint32_t ncodes = 0, nlits = 0;
        if (K == E_MIO0 || K == E_YAY0) {
            // worst case: n literal bytes, n/3*2 code bytes (+ n/18 extended lengths counted in lits)
            codes = reinterpret_cast<uint8_t*>(f.head) + P.scratch_per_warp - 2 * (size_t(n) + 64);
            lits = codes + size_t(n) + 32;
        }

        // ---- headers
        // BLZ.cs:143-215: CompressHeaderless over the (already reversed) source — LZ10's flag / token layout without a header,
        // distance - 3 in the code; the host side reverses the code stream and appends padding + footer
        const bool blz = K == E_LZ10 && P.format == AURORA_FMT_BLZ;
        const bool lz40 = K == E_LZ11 && (P.format == AURORA_FMT_LZ40 || P.format == AURORA_FMT_LZ60);   // LZ40.cs:126-168
        if (blz) {
            // no header
        } else if (K == E_LZ10 || K == E_LZ11) {
            const uint32_t id = K == E_LZ10 ? 0x10 : !lz40 ? 0x11 : P.format == AURORA_FMT_LZ40 ? 0x40 : 0x60;
            w.negate = lz40;
            if (n <= 0xFFFFFF) {
                put_u32(w, id | (uint32_t(n) << 8), false);
            } else {
                put_u32(w, id, false);
                put_u32(w, uint32_t(n), false);
            }
        } else if (K == E_YAZ0 && P.format == AURORA_FMT_LZHUDSON) {
            // LZHudson.cs:48-59: u32 BE size, then Yay0.CompressHeaderless under FlagWriter(destination, Endian.Big, 4, Endian.Big)
            put_u32(w, uint32_t(n), true);
            w.flag_bytes = 4;
        } else if (K == E_YAZ0) {
            const char* magic = P.format == AURORA_FMT_YAZ1 ? "Yaz1" : "Yaz0";
            for (int i = 0; i < 4; i++) w.raw_byte(uint8_t(magic[i]));
            put_u32(w, uint32_t(n), big);
            put_u32(w, P.yaz0_alignment, big);
            put_u32(w, 0, false);
        } else if (K == E_LZSS) {
            w.raw_byte('L'); w.raw_byte('Z'); w.raw_byte('S'); w.raw_byte('S');
            put_u32(w, uint32_t(n), true);
            put_u32(w, 0, false);   // compressed size, patched below
            put_u32(w, 0, false);
        } else if (K == E_MIO0 && P.format == AURORA_FMT_SMSR00) {
            // SMSR00.cs:60-75: "SMSR00", u16 0, BE size, BE pointer to the literal section (patched below); the code section is
            // MIO0.CompressHeaderless under FlagWriter(codeData, Endian.Big, 2, Endian.Big) with the codes in its buffer
            const char* magic = "SMSR00";
            for (int i = 0; i < 6; i++) w.raw_byte(uint8_t(magic[i]));
            w.raw_byte(0);
            w.raw_byte(0);
            put_u32(w, uint32_t(n), true);
            put_u32(w, 0, true);
            w.flag_bytes = 2;
        } else {
            const char* magic = K == E_MIO0 ? "MIO0" : "Yay0";
            for (int i = 0; i < 4; i++) w.raw_byte(uint8_t(magic[i]));
            put_u32(w, uint32_t(n), big);
            put_u32(w, 0, big);   // offsets patched below
            put_u32(w, 0, big);
        }
        const uint64_t body_start = w.pos;

        // ---- token loop (the common shape of all CompressHeaderless bodies)
        const int lz_n = P.lzss.max_distance - 1, lz_f = (1 << P.lzss.length_bits) - 1;
        int sp = 0;
        for (;;) {
            const Match m = find_next_best_match(f, src, n);
            int plain = m.offset - sp;
            while (plain != 0) {
                plain--;
                const uint32_t b = src[sp++];
                if (K == E_MIO0 || K == E_YAY0) {
                    if (lane == 0) lits[nlits] = uint8_t(b);
                    nlits++;
                    w.bit(true);
                } else {
                    w.byte(b);
                    w.bit(K == E_YAZ0 || K == E_LZSS);   // Yaz0/LZSS: 1 = literal; LZ10/LZ11: 0 = literal
                }
            }
            if (m.length == 0) break;
            const uint32_t d1 = uint32_t(m.distance - 1) & 0xFFF;
            if (K == E_LZ10) {
                const uint32_t v = uint32_t(m.length - 3) << 12 | (blz ? uint32_t(m.distance - 3) & 0xFFF : d1);
                w.byte((v >> 8) & 0xFF);
                w.byte(v & 0xFF);
                w.bit(true);
            } else if (K == E_LZ11 && lz40) {
                // (ushort)(Distance << 4 | ...), little-endian: a distance of 0x1000 truncates to 0
                const uint32_t dd = (uint32_t(m.distance) << 4) & 0xFFFF;
                if (m.length < 16) {
                    w.byte((dd | uint32_t(m.length)) & 0xFF);
                    w.byte(dd >> 8);
                } else if (m.length < 272) {
                    w.byte(dd & 0xFF);
                    w.byte(dd >> 8);
                    w.byte(uint32_t(m.length - 16) & 0xFF);
                } else {
                    w.byte((dd | 1u) & 0xFF);
                    w.byte(dd >> 8);
                    w.byte(uint32_t(m.length - 272) & 0xFF);
                    w.byte((uint32_t(m.length - 272) >> 8) & 0xFF);
                }
                w.bit(true);
            } else if (K == E_LZ11) {
                if (m.length <= 16) {
                    const uint32_t v = (uint32_t(m.length - 1) << 12 | d1) & 0xFFFF;
                    w.byte(v >> 8);
                    w.byte(v & 0xFF);
                } else if (m.length <= 272) {
                    w.byte((uint32_t(m.length - 17) & 0xFF) >> 4);
                    const uint32_t v = (uint32_t(m.length - 17) << 12 | d1) & 0xFFFF;
                    w.byte(v >> 8);
                    w.byte(v & 0xFF);
                } else {
                    const uint32_t v = 0x10000000u | (uint32_t(m.length - 273) & 0xFFFF) << 12 | d1;
                    w.byte(v >> 24);
                    w.byte((v >> 16) & 0xFF);
                    w.byte((v >> 8) & 0xFF);
                    w.byte(v & 0xFF);
                }
                w.bit(true);
            } else if (K == E_YAZ0) {
                if (m.length < 18) {
                    const uint32_t v = (uint32_t(m.distance - 1) | uint32_t(m.length - 2) << 12) & 0xFFFF;
                    w.byte(v >> 8);
                    w.byte(v & 0xFF);
                } else {
                    w.byte(d1 >> 8);
                    w.byte(d1 & 0xFF);
                    w.byte(uint32_t(m.length - 0x12) & 0xFF);
                }
                w.bit(false);
            } else if (K == E_LZSS) {
                const int offset = (P.lzss.windows_start + sp - m.distance) & lz_n;
                const uint32_t v = (uint32_t(offset & 0xFF) | uint32_t(offset & 0xFF00) << P.lzss.length_bits |
                                    uint32_t((m.length - P.lzss.min_length) & lz_f) << 8) & 0xFFFF;
                w.byte(v & 0xFF);
                w.byte(v >> 8);
                w.bit(false);
            } else {   // MIO0 / Yay0 codes go to their own section
                uint32_t v;
                if (K == E_MIO0) v = (uint32_t(m.distance - 1) | uint32_t(m.length - 3) << 12) & 0xFFFF;
                else if (m.length < 18) v = (uint32_t(m.distance - 1) | uint32_t(m.length - 2) << 12) & 0xFFFF;
                else v = d1;
                if (K == E_MIO0 && P.format == AURORA_FMT_SMSR00) {   // the codes share the section of their mask words
                    w.byte(v >> 8);
                    w.byte(v & 0xFF);
                } else {
                    if (lane == 0) {
                        codes[ncodes] = uint8_t(v >> 8);
                        codes[ncodes + 1] = uint8_t(v & 0xFF);
                    }
                    ncodes += 2;
                }
                if (K == E_YAY0 && m.length >= 18) {
                    if (lane == 0) lits[nlits] = uint8_t(m.length - 0x12);
                    nlits++;
                }
                w.bit(false);
            }
            sp += m.length;
        }
        if (K == E_MIO0 || K == E_YAY0) {
            // the flag section holds only flag bytes: the Writer reserved one byte per group and wrote nothing else
            w.dispose();
            __syncwarp();
            const uint64_t comp_off = w.pos, lit_off = w.pos + ncodes;
            for (uint32_t i = lane; i < ncodes; i += 32)
                if (comp_off + i < w.cap) w.out[comp_off + i] = codes[i];
            for (uint32_t i = lane; i < nlits; i += 32)
                if (lit_off + i < w.cap) w.out[lit_off + i] = lits[i];
            w.pos = lit_off + nlits;
            if (w.pos > w.cap) w.overflow = true;
            const uint64_t save = w.pos;
            if (K == E_MIO0 && P.format == AURORA_FMT_SMSR00) {
                w.pos = 12;
                put_u32(w, uint32_t(lit_off), true);   // ncodes == 0: the literal section starts where the code section ends
            } else {
                w.pos = 8;
                put_u32(w, uint32_t(comp_off), big);
                put_u32(w, uint32_t(lit_off), big);
            }
            w.pos = save;
        } else {
            w.dispose();
            if (K == E_LZSS) {
                const uint64_t save = w.pos;
                w.pos = 8;
                put_u32(w, uint32_t(save - body_start), true);
                w.pos = save;
            }
        }
        out_len = w.pos;
        if (w.overflow) status = AURORA_DST_TOO_SMALL;
    }
    if (lane == 0) {
        P.out_len[idx] = out_len;
        P.status[idx] = status;
    }
    __syncwarp();
}

// ---- kernel
template <int K>
__global__ void __launch_bounds__(kEncWarpsPerBlock * 32) encode_lz_kernel(const EncodeParams P) {
    const int warp_global = blockIdx.x * kEncWarpsPerBlock + (threadIdx.x >> 5);
    uint8_t* scratch = P.scratch + size_t(warp_global) * P.scratch_per_warp;
    Finder f;
    finder_setup(f, P, scratch);
    for (;;) {
        uint32_t t = 0;
        if (lane_id() == 0) t = atomicAdd(P.ticket, 1u);
        t = __shfl_sync(kFull, t, 0);
        if (t >= P.n) break;
        encode_stream<K>(P, t, f);
    }
}

template <int K>
cudaError_t launch(const EncodeParams& p, int warps, cudaStream_t st) {
    encode_lz_kernel<K><<<warps / kEncWarpsPerBlock, kEncWarpsPerBlock * 32, 0, st>>>(p);
    return cudaGetLastError();
}

}  // namespace

int encode_resident_warps(int sm_count) { return sm_count * 48; }

// head + chain + min tables, plus (MIO0/Yay0) staging for the code and literal sections
size_t encode_scratch_per_warp(int format, int hash_bits, int chain_bits, uint64_t max_src_len) {
    size_t bytes = (size_t(1) << hash_bits) * 4 + (size_t(1) << chain_bits) * 4 + 65536 * 4;
    if (format == AURORA_FMT_MIO0 || format == AURORA_FMT_YAY0 || format == AURORA_FMT_SMSR00) bytes += 2 * (size_t(max_src_len) + 64);
    return (bytes + 255) & ~size_t(255);
}

cudaError_t launch_encode_lz(const EncodeParams& p, int warps, cudaStream_t st) {
    switch (p.format) {
        case AURORA_FMT_LZ10:
        case AURORA_FMT_BLZ: return launch<E_LZ10>(p, warps, st);   // BLZ: LZ10's layout over the reversed source, distance - 3
        case AURORA_FMT_LZ11:
        case AURORA_FMT_LZ40:
        case AURORA_FMT_LZ60: return launch<E_LZ11>(p, warps, st);   // LZ40 / LZ60: the LZ11 parse with LE tokens and negated flags
        case AURORA_FMT_YAZ0:
        case AURORA_FMT_YAZ1:
        case AURORA_FMT_LZHUDSON: return launch<E_YAZ0>(p, warps, st);   // the same tokens under 4-byte flag words
        case AURORA_FMT_LZSS: return launch<E_LZSS>(p, warps, st);
        case AURORA_FMT_MIO0:
        case AURORA_FMT_SMSR00: return launch<E_MIO0>(p, warps, st);   // SMSR00: MIO0 tokens, 16-bit masks interleaved with the codes
        case AURORA_FMT_YAY0: return launch<E_YAY0>(p, warps, st);
        default: return cudaErrorNotSupported;
    }
}

}  // namespace aurora
