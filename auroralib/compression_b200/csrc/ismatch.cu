// ismatch.cu — the IsMatch and GetDecompressedSize rules of the core formats (SURVEY.md Appendix A "IsMatch rules"), written
// once.  is_match_one is __host__ __device__: the library runs the magic / footer rules on the host (a peek of a few bytes)
// and the token walks on the device, where the IsMatch and offset-scan kernels call it for every format.
// The token walks are LZ10.Validate (Nintendo/LZ10.cs:139-175), LZ11.Validate (LZ11.cs:173-223) and PRS.GetByteOrder /
// ValidateByteOrder (Sega/PRS.cs:161-218).  They stop at the 4th plausible match, so they are short and independent: one THREAD
// per candidate stream, reading the blob straight from global memory (this is the data-parallel form of the CLI's
// byte-by-byte `-scan` loop, Commands/ScanDecompressCommand.cs:23-39).  An exception inside the reference's walk (a read past
// the end) makes IsMatch false here, like the oracle.
// core_decoded_size (size_peek.cuh) and decoded_size_one are __host__ __device__ too: aurora_decoded_size_batch runs them on the host,
// aurora_decoded_size_batch_device in decoded_size_kernel, one thread per stream.
// launch_window_hits (at the end) selects the hits of one window of aurora_scan_decode_device's walk with the same rule.
#include "api_internal.hpp"
#include "common.cuh"
#include "size_peek.cuh"

namespace aurora {

namespace {

struct BitReader {   // FlagReader with a 1-byte flag word (IO/FlagReader.cs:53-65)
    const uint8_t* p;
    uint64_t len, pos;
    uint32_t cur, left;
    bool msb, fail;
    __host__ __device__ int bit() {
        if (left == 0) {
            if (pos >= len) { fail = true; return 0; }
            cur = p[pos++];
            left = 8;
        }
        const uint32_t sh = msb ? left - 1 : 8 - left;
        left--;
        return (cur >> sh) & 1;
    }
    __host__ __device__ uint32_t byte() {
        if (pos >= len) { fail = true; return 0; }
        return p[pos++];
    }
};

__host__ __device__ bool lz1x_validate(const uint8_t* p, uint64_t len, bool lz11) {
    if (!(8 < len)) return false;   // stream.Position + 0x8 < stream.Length
    if (p[0] != (lz11 ? 0x11 : 0x10)) return false;
    uint64_t pos = 4;
    uint32_t size = uint32_t(p[1]) | (uint32_t(p[2]) << 8) | (uint32_t(p[3]) << 16);
    if (size == 0) {
        size = uint32_t(p[4]) | (uint32_t(p[5]) << 8) | (uint32_t(p[6]) << 16) | (uint32_t(p[7]) << 24);
        pos = 8;
    }
    if (size == 0) return false;
    int budget = 3;
    uint64_t produced = 0;
    BitReader r{p, len, pos, 0, 0, true, false};
    while (r.pos < len) {
        const int b = r.bit();
        if (r.fail) return false;
        if (b) {
            uint32_t distance, length;
            const uint32_t b1 = r.byte(), b2 = r.byte();
            if (lz11 && (b1 >> 4) == 0) {
                const uint32_t b3 = r.byte();
                distance = (((b2 & 0xf) << 8) | b3) + 1;
                length = (((b1 & 0xf) << 4) | (b2 >> 4)) + 17;
            } else if (lz11 && (b1 >> 4) == 1) {
                const uint32_t b3 = r.byte(), b4 = r.byte();
                distance = (((b3 & 0xf) << 8) | b4) + 1;
                length = (((b1 & 0xf) << 12) | (b2 << 4) | (b3 >> 4)) + 273;
            } else {
                distance = (((b1 & 0xf) << 8) | b2) + 1;
                length = (b1 >> 4) + (lz11 ? 1 : 3);
            }
            if (r.fail) return false;
            if (distance > produced) return false;
            if (budget == 0) return true;
            budget--;
            produced += length;
        } else {
            r.pos++;   // source.Position++ (no bounds check in the reference)
            produced++;
        }
    }
    return produced == size;
}

// 1 valid, 0 invalid, -1 exception
__host__ __device__ int prs_validate(const uint8_t* p, uint64_t len, bool big) {
    int budget = 3;
    uint64_t produced = 0;
    BitReader r{p, len, 0, 0, 0, big, false};
    while (r.pos < len) {
        int b = r.bit();
        if (r.fail) return -1;
        if (b) {
            r.pos++;
            produced++;
        } else {
            uint32_t distance, length;
            b = r.bit();
            if (r.fail) return -1;
            if (b) {
                if (r.pos + 2 > len) return -1;
                const uint32_t v = big ? (uint32_t(p[r.pos]) << 8) | p[r.pos + 1] : uint32_t(p[r.pos]) | (uint32_t(p[r.pos + 1]) << 8);
                r.pos += 2;
                if (v == 0) return 1;
                length = v & 7;
                distance = 0x2000 - (v >> 3);
                if (length == 0) {
                    length = r.byte() + 1;
                    if (r.fail) return -1;
                } else {
                    length += 2;
                }
            } else {
                const int b1 = r.bit(), b0 = r.bit();
                if (r.fail) return -1;
                length = uint32_t(b1 * 2 + b0) + 2;
                distance = 0x100 - r.byte();
                if (r.fail) return -1;
            }
            if (distance > produced) return 0;
            if (budget == 0) return 1;
            budget--;
            produced += length;
        }
    }
    return 0;
}

}  // namespace

__host__ __device__ int is_match_one(const uint8_t* p, uint64_t len, int format) {
    auto magic = [&](uint32_t be) {
        return 0x10 < len && ((uint32_t(p[0]) << 24) | (uint32_t(p[1]) << 16) | (uint32_t(p[2]) << 8) | p[3]) == be;
    };
    switch (format) {
        case AURORA_FMT_YAZ0: return magic(0x59617A30u);
        case AURORA_FMT_YAZ1: return magic(0x59617A31u);
        case AURORA_FMT_LZHUDSON: return 0x8 < len && (p[0] | p[1] | p[2] | p[3]) != 0;   // LZHudson.cs:31-32, no file name
        case AURORA_FMT_SMSR00:   // SMSR00.cs:36-37
            return 0x10 < len && p[0] == 'S' && p[1] == 'M' && p[2] == 'S' && p[3] == 'R' && p[4] == '0' && p[5] == '0';
        case AURORA_FMT_LZ40:   // LZ40.cs:41-43, LZ60.cs:31-33: identifier and a non-zero size ("recognition is inaccurate!")
        case AURORA_FMT_LZ60:
            return 0x8 < len && p[0] == (format == AURORA_FMT_LZ40 ? 0x40 : 0x60) && ((p[1] | p[2] | p[3]) != 0 || (p[4] | p[5] | p[6] | p[7]) != 0);
        case AURORA_FMT_YAY0: return magic(0x59617930u);
        case AURORA_FMT_MIO0: return magic(0x4D494F30u);
        case AURORA_FMT_LZSS: return magic(0x4C5A5353u);
        case AURORA_FMT_LZ4_LEGACY: return magic(0x02214C18u);
        case AURORA_FMT_LZ4: {
            if (!(0x10 < len)) return false;
            const uint32_t v = uint32_t(p[0]) | (uint32_t(p[1]) << 8) | (uint32_t(p[2]) << 16) | (uint32_t(p[3]) << 24);
            return v == 0x184C2102u || v == 0x184D2204u || (v >= 0x184D2A50u && v <= 0x184D2A5Fu);
        }
        case AURORA_FMT_SNAPPY: {
            const uint8_t id[10] = {0xff, 0x06, 0x00, 0x00, 0x73, 0x4e, 0x61, 0x50, 0x70, 0x59};
            if (!(0x10 < len)) return false;
            for (int i = 0; i < 10; i++)
                if (p[i] != id[i]) return false;
            return true;
        }
        case AURORA_FMT_LZO: return len > 0 && p[0] < 0x20;   // LZO.cs:31-39 without a file name
        case AURORA_FMT_LZ10: return lz1x_validate(p, len, false);
        case AURORA_FMT_LZ11: return lz1x_validate(p, len, true);
        case AURORA_FMT_PRS: {
            if (!(4 < len)) return false;   // stream.Position + 0x4 < stream.Length
            const uint32_t flag = p[0];
            int v = 0;
            if (flag > 12 && (flag & 1)) v = prs_validate(p, len, false);
            if (v == 0 && (flag & 128)) v = prs_validate(p, len, true);
            return v == 1;
        }
        case AURORA_FMT_BLZ:   // BLZ.cs:31-32: the footer's compressed size is the whole stream, footer size >= 8
            return len >= 8 && (uint64_t(p[len - 8]) | (uint64_t(p[len - 7]) << 8) | (uint64_t(p[len - 6]) << 16)) == len && p[len - 5] >= 8;
    }
    return -1;
}

__host__ __device__ int decoded_size_one(int format, int byte_order, const uint8_t* p, uint64_t len, uint64_t* size) {
    if (is_bytelz(format)) {   // LZ4 / LZO / Snappy / PRS do not implement IProvidesDecompressedSize
        *size = 0;
        return AURORA_NOT_SUPPORTED;
    }
    return core_decoded_size(format, byte_order, p, len, size);
}

__host__ __device__ int size_scan_status(int status) {
    // the scan decodes against a zero capacity: a stream that parses to its end reports DST_TOO_SMALL
    return status == AURORA_DST_TOO_SMALL ? AURORA_OK : status;
}

// ---- kernel
namespace {

__global__ void is_match_kernel(const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len, uint8_t* match, uint32_t n, int format) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    match[i] = is_match_one(src_base + src_off[i], src_len[i], format) > 0;
}

// Offset scan: IsMatch at EVERY byte offset of one image (the data-parallel form of the CLI's `-scan` loop,
// Commands/ScanDecompressCommand.cs:23-39): thread i tests the stream that starts at offset i and runs to the end.
__global__ void scan_kernel(const uint8_t* image, uint64_t len, uint8_t* match, int format) {
    const uint64_t i = uint64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= len) return;
    match[i] = is_match_one(image + i, len - i, format) > 0;
}

__global__ void decoded_size_kernel(const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len, uint64_t* size,
                                    int32_t* status, uint32_t n, int format, int byte_order) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t s;
    status[i] = decoded_size_one(format, byte_order, src_base + src_off[i], src_len[i], &s);
    size[i] = s;
}

__global__ void size_scan_status_kernel(int32_t* status, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) status[i] = size_scan_status(status[i]);
}

// ---- largest-first stream order for batches with a wide size spread: counting sort by floor(log2(size)) ----
__global__ void order_hist_kernel(const uint64_t* size, uint32_t n, uint32_t* hist) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicAdd(&hist[63 - __clzll((long long)(size[i] | 1))], 1u);
}
__global__ void order_scan_kernel(uint32_t* hist) {   // one thread: descending exclusive offsets over 64 buckets
    uint32_t acc = 0;
    for (int b = 63; b >= 0; b--) {
        const uint32_t c = hist[b];
        hist[b] = acc;
        acc += c;
    }
}
__global__ void order_scatter_kernel(const uint64_t* size, uint32_t n, uint32_t* hist, uint32_t* order) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) order[atomicAdd(&hist[63 - __clzll((long long)(size[i] | 1))], 1u)] = i;
}

}  // namespace

cudaError_t launch_size_order(const uint64_t* d_size, uint32_t n, uint32_t* d_hist64, uint32_t* d_order, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(d_hist64, 0, 64 * sizeof(uint32_t), st);
    if (e != cudaSuccess) return e;
    order_hist_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_size, n, d_hist64);
    order_scan_kernel<<<1, 1, 0, st>>>(d_hist64);
    order_scatter_kernel<<<(n + 255) / 256, 256, 0, st>>>(d_size, n, d_hist64, d_order);
    return cudaGetLastError();
}

cudaError_t launch_scan(const uint8_t* image, uint64_t len, uint8_t* match, int format, cudaStream_t st) {
    scan_kernel<<<uint32_t((len + 255) / 256), 256, 0, st>>>(image, len, match, format);
    return cudaGetLastError();
}

cudaError_t launch_is_match(const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len, uint8_t* match, uint32_t n,
                            int format, cudaStream_t st) {
    is_match_kernel<<<(n + 127) / 128, 128, 0, st>>>(src_base, src_off, src_len, match, n, format);
    return cudaGetLastError();
}

cudaError_t launch_decoded_size(const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len, uint64_t* size,
                                int32_t* status, uint32_t n, int format, int byte_order, cudaStream_t st) {
    decoded_size_kernel<<<(n + 127) / 128, 128, 0, st>>>(src_base, src_off, src_len, size, status, n, format, byte_order);
    return cudaGetLastError();
}

cudaError_t launch_size_scan_status(int32_t* status, uint32_t n, cudaStream_t st) {
    size_scan_status_kernel<<<(n + 255) / 256, 256, 0, st>>>(status, n);
    return cudaGetLastError();
}

}  // namespace aurora

// ---- the hits of one window of the offset walk (aurora_scan_decode_device, scan_decode.cu)
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/tabulate_output_iterator.h>

namespace aurora {

namespace {

struct WindowHit {   // IsMatch of the stream at *base + i, to the end of the image (*base: the round's walk position)
    const uint8_t* image;
    uint64_t len;
    const uint64_t* base;
    int format;
    __device__ bool operator()(uint32_t i) const {
        const uint64_t q = *base + i;
        return q < len && is_match_one(image + q, len - q, format) > 0;
    }
};

struct KeepFirst {   // the select's output: only the first `keep` hits are stored, all of them are counted
    uint32_t* out;
    uint32_t keep;
    template <typename I>
    __device__ void operator()(I idx, uint32_t v) const {
        if (uint64_t(idx) < keep) out[idx] = v;
    }
};

}  // namespace

cudaError_t launch_window_hits(const uint8_t* image, uint64_t len, const uint64_t* d_base, uint32_t items, int format, uint32_t* rel,
                               uint32_t keep, uint32_t* d_count, void* temp, size_t* temp_bytes, cudaStream_t st) {
    return cub::DeviceSelect::If(temp, *temp_bytes, thrust::counting_iterator<uint32_t>(0),
                                 thrust::make_tabulate_output_iterator(KeepFirst{rel, keep}), d_count, int64_t(items),
                                 WindowHit{image, len, d_base, format}, st);
}

}  // namespace aurora
