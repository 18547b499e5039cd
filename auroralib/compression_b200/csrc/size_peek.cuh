// size_peek.cuh — core_decoded_size, the one copy of the GetDecompressedSize header peek of BLZ and the flag-LZ formats.  A
// header, because device code in two translation units calls it: decoded_size_kernel (ismatch.cu) and the ChunkLZ10 chunk
// walk of the wrapper kernels (wrappers.cu).  A status; *size is 0 unless it is AURORA_OK.  AURORA_INVALID_ARGUMENT for a
// format without a size header.
#pragma once
#include <stdint.h>

#include "../../../include/aurora_cuda.h"

namespace aurora {

__host__ __device__ inline int core_decoded_size(int format, int byte_order, const uint8_t* p, uint64_t len, uint64_t* size) {
    auto be32 = [](const uint8_t* q) { return (uint32_t(q[0]) << 24) | (uint32_t(q[1]) << 16) | (uint32_t(q[2]) << 8) | q[3]; };
    auto le32 = [](const uint8_t* q) { return uint32_t(q[0]) | (uint32_t(q[1]) << 8) | (uint32_t(q[2]) << 16) | (uint32_t(q[3]) << 24); };
    *size = 0;
    switch (format) {
        case AURORA_FMT_BLZ: {   // BLZ.cs:35-43: the footer at Length - 8
            if (len < 8) return AURORA_END_OF_STREAM;
            const uint8_t* f = p + len - 8;
            if (f[3] < 8) return AURORA_INVALID_DATA;   // "Invalid BLZ header."
            *size = uint32_t(le32(f + 4) + (uint32_t(f[0]) | (uint32_t(f[1]) << 8) | (uint32_t(f[2]) << 16)));
            return AURORA_OK;
        }
        case AURORA_FMT_LZHUDSON:   // LZHudson.cs:37-38
            if (len < 4) return AURORA_END_OF_STREAM;
            *size = be32(p);
            return AURORA_OK;
        case AURORA_FMT_SMSR00:   // SMSR00.cs:40-46
            if (len < 6) return AURORA_END_OF_STREAM;
            for (int k = 0; k < 6; k++)
                if (p[k] != uint8_t("SMSR00"[k])) return AURORA_INVALID_IDENTIFIER;
            if (len < 12) return AURORA_END_OF_STREAM;
            *size = be32(p + 8);
            return AURORA_OK;
        case AURORA_FMT_LZ10: case AURORA_FMT_LZ11: case AURORA_FMT_LZ40: case AURORA_FMT_LZ60: {   // LZ10.cs:47-57: type byte + u24, u32 when 0
            const uint8_t id = format == AURORA_FMT_LZ10 ? 0x10 : format == AURORA_FMT_LZ11 ? 0x11 : format == AURORA_FMT_LZ40 ? 0x40 : 0x60;
            if (len < 1) return AURORA_END_OF_STREAM;
            if (p[0] != id) return AURORA_INVALID_IDENTIFIER;
            if (len < 4) return AURORA_END_OF_STREAM;
            uint32_t v = uint32_t(p[1]) | (uint32_t(p[2]) << 8) | (uint32_t(p[3]) << 16);
            if (v == 0) {
                if (len < 8) return AURORA_END_OF_STREAM;
                v = le32(p + 4);
            }
            *size = v;
            return AURORA_OK;
        }
        case AURORA_FMT_YAZ0: case AURORA_FMT_YAZ1: case AURORA_FMT_YAY0: case AURORA_FMT_MIO0: case AURORA_FMT_LZSS: {   // e.g. Yaz0.cs:50-55
            const char* magic = format == AURORA_FMT_YAZ0 ? "Yaz0" : format == AURORA_FMT_YAZ1 ? "Yaz1" : format == AURORA_FMT_YAY0 ? "Yay0"
                                : format == AURORA_FMT_MIO0 ? "MIO0" : "LZSS";
            if (len < 4) return AURORA_END_OF_STREAM;
            for (int k = 0; k < 4; k++)
                if (p[k] != uint8_t(magic[k])) return AURORA_INVALID_IDENTIFIER;
            if (len < 8) return AURORA_END_OF_STREAM;
            bool big = true;   // LZSS, and Yay0.cs:45-46 reads BE regardless
            if (format == AURORA_FMT_YAZ0 || format == AURORA_FMT_YAZ1) {
                big = byte_order != AURORA_ENDIAN_LITTLE;
            } else if (format == AURORA_FMT_MIO0) {   // MIO0.cs:42-48: detected order
                if (byte_order == AURORA_ENDIAN_LITTLE) big = false;
                else if (byte_order != AURORA_ENDIAN_BIG && len >= 16) {
                    const uint32_t cb = be32(p + 8), lb = be32(p + 12), cl = le32(p + 8), ll = le32(p + 12);
                    const bool pb = cb >= 0x10 && cb <= lb && lb <= len, pl = cl >= 0x10 && cl <= ll && ll <= len;
                    big = pb || !pl;
                }
            }
            *size = big ? be32(p + 4) : le32(p + 4);
            return AURORA_OK;
        }
    }
    return AURORA_INVALID_ARGUMENT;
}

}  // namespace aurora
