// common.cuh — shared device/host definitions for libaurora_cuda.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../../include/aurora_cuda.h"

namespace aurora {

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xFFFFFFFFu;

// LZSS parameters resolved on the host from aurora_lz_props (LzProperties.cs)
struct LzssParams {
    int windows_bits, length_bits, min_length, max_distance, windows_start, initial_fill;
};

// One batch on one device.  All pointers are device pointers.
struct DecodeParams {
    const uint8_t* src_base;
    uint64_t src_limit;          // readable bytes from src_base, a multiple of 16 (TMA bulk granularity)
    const uint64_t* src_off;
    const uint64_t* src_len;
    uint8_t* dst_base;
    const uint64_t* dst_off;
    const uint64_t* dst_cap;
    uint64_t* out_len;
    uint64_t* consumed;
    int32_t* status;
    const uint32_t* order;       // optional: stream indices, largest first (nullptr = identity)
    unsigned int* ticket;        // global work counter (zeroed by the launcher)
    uint32_t n;
    int format;
    int byte_order;              // aurora_endian
    int size_only;               // parse without copying (decoded_size_batch size_scan)
    int lz4_verify;              // LZ4.HashAlgorithm set: verify XXH32 checksums
    int headerless;              // LZ10/LZ11/LZSS DecompressHeaderless(source, destination, size): the stream is the bare token
                                 // body and dst_cap[i] carries (size << 32) | min(capacity, 2^32 - 1)  (wrapper formats)
    LzssParams lzss;
};

struct EncodeParams {
    const uint8_t* src_base;
    uint64_t src_limit;
    const uint64_t* src_off;
    const uint64_t* src_len;
    uint8_t* dst_base;
    const uint64_t* dst_off;
    const uint64_t* dst_cap;
    uint64_t* out_len;
    int32_t* status;
    unsigned int* ticket;
    uint32_t n;
    int format;
    int byte_order;
    // CompressionSettings -> LzChainMatchFinder parameters (LzChainMatchFinder.cs:108-119)
    int max_chain, lazy_threshold, hash_bits, chain_bits, min_length, max_length, min_distance, max_distance, no_self_overlap,
        use_min_table;
    int finder_choice;   // 0 automatic, 1 one lane per window position (encode_lz_par.cu), 2 sequential replay (finder.cuh)
    uint32_t yaz0_alignment;
    uint32_t lz4_block_size;
    LzssParams lzss;
    uint8_t* scratch;            // per-resident-warp match-finder tables
    uint64_t scratch_per_warp;
};

// aurora_encode_bound of the core formats: the worst case of every token writer on the hot path, all literals + flag bits +
// headers / chunk framing (also the chunk slots of a ChunkLZ10 encode, wrappers.cu)
__host__ __device__ inline uint64_t core_encode_bound(int format, uint64_t raw_len) {
    switch (format) {
        case AURORA_FMT_LZ4:
        case AURORA_FMT_LZ4_LEGACY:
        case AURORA_FMT_LZ4_BLOCK: return raw_len + raw_len / 255 + 64 + 8 * (raw_len / 0x400000 + 1);
        case AURORA_FMT_SNAPPY:
        case AURORA_FMT_SNAPPY_BLOCK: return raw_len + raw_len / 60 + 32 + 16 * (raw_len / 0x10000 + 1);
        // LZO: a far 3-byte match costs 3 bytes and splits the literal run around it (4 literals + 1 match = 7 bytes in, 8 out)
        case AURORA_FMT_LZO: return raw_len + raw_len / 6 + 64;
        // LZSS with min_length 1: a two-byte token for each input byte, and a flag byte per 8 tokens
        case AURORA_FMT_LZSS: return 2 * raw_len + raw_len / 8 + 64;
        default: return raw_len + raw_len / 8 + 64;
    }
}

#ifdef __CUDACC__   // (not in the CPU builds of the kernel sources under tests/simt)
// a device allocation that grows (never shrinks) to the largest request; cudaFree of the old block synchronises the device
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = n + n / 8 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// per-device scratch of aurora_decode_batch_device / aurora_encode_batch_device for the wrapper formats (wrappers.cu):
// per-stream plans and sub-streams (+ LZ77's chunk counts and scan), the core launches' descriptors and results, LZ00's
// keystream-free bodies (decode: one 16-byte aligned slot per stream)
struct WrapScratch {
    DevBuf plans, slots, src;
    void release() {
        plans.release();
        slots.release();
        src.release();
    }
};
// the wrapper pipeline on the caller's device arrays; counts its kernel launches into *launches
cudaError_t wrapped_decode_batch_device(int format, const aurora_codec_opts* opts, size_t n, const uint8_t* d_src_base, uint64_t src_total,
                                        const uint64_t* d_src_off, const uint64_t* d_src_len, uint8_t* d_dst_base,
                                        const uint64_t* d_dst_off, const uint64_t* d_dst_cap, uint64_t* d_out_len,
                                        uint64_t* d_consumed, int32_t* d_status, WrapScratch& scr, unsigned int* ticket, int sm_count,
                                        cudaStream_t st, uint64_t* launches);
// the wrapper encode pipeline on the caller's device arrays (enc_scratch: the core encoder's per-warp tables); returns
// AURORA_OK, AURORA_INVALID_ARGUMENT (settings) or AURORA_CUDA_ERROR with *err set; counts its kernel launches into *launches
int wrapped_encode_batch_device(int format, const aurora_codec_opts* opts, size_t n, const uint8_t* d_src_base, uint64_t src_total,
                                const uint64_t* d_src_off, const uint64_t* d_src_len, uint8_t* d_dst_base, const uint64_t* d_dst_off,
                                const uint64_t* d_dst_cap, uint64_t* d_out_len, int32_t* d_status, WrapScratch& scr,
                                DevBuf& enc_scratch, unsigned int* ticket, int sm_count, cudaStream_t st, uint64_t* launches,
                                cudaError_t* err);
#endif

// api.cu: the option block resolved into kernel parameters (returns a per-batch status override, OK = run), and the decode
// kernel of p.format
int fill_decode_params(DecodeParams& p, int format, const aurora_codec_opts* o);
cudaError_t launch_decode(const DecodeParams& p, int sm_count, cudaStream_t st);
// the same for the encoders: CompressionSettings + LzProperties -> finder parameters (AURORA_OK, or the batch's argument
// error), and the encode kernel of p.format (the lane-per-position finder or the sequential replay)
int fill_encode_params(EncodeParams& p, int format, const aurora_codec_opts* o);
// The warps launch_encode starts for the p.n streams of a batch: one per stream, up to the resident warps of the encoder it
// picks.  Each of them owns one slice of p.scratch, so the scratch reservation takes this count as well.
int encode_launch_warps(const EncodeParams& p, int sm_count);
// The sequential replay's chain table for streams of at most `longest` bytes (see api.cu)
int encode_chain_bits(int chain_bits, uint64_t longest);
cudaError_t launch_encode(const EncodeParams& p, int warps, cudaStream_t st);
// kernel launchers (one translation unit per kernel family); all return cudaGetLastError()
cudaError_t launch_decode_flaglz(const DecodeParams& p, int sm_count, cudaStream_t st);
cudaError_t launch_decode_bytelz(const DecodeParams& p, int sm_count, cudaStream_t st);
cudaError_t launch_decode_blz(const DecodeParams& p, int sm_count, cudaStream_t st);
// in-place byte reversal of bytes [0, min(len[i], cap[i])) of every stream (BLZ encode; decode_blz.cu); cap may be null
cudaError_t launch_reverse_bytes(uint8_t* base, const uint64_t* d_off, const uint64_t* d_len, const uint64_t* d_cap, uint32_t n,
                                 cudaStream_t st);
constexpr int kEncWarpsPerBlock = 8;   // the sequential replay (encode_lz.cu, encode_bytelz.cu); `warps`: a multiple of it
cudaError_t launch_encode_lz(const EncodeParams& p, int warps, cudaStream_t st);
cudaError_t launch_encode_bytelz(const EncodeParams& p, int warps, cudaStream_t st);
bool encode_lz_par_supported(const EncodeParams& p);   // encode_lz_par.cu: one lane per window position
int encode_lz_par_block_warps(const EncodeParams& p);  // its warps per block (one block per SM)
cudaError_t launch_encode_lz_par(const EncodeParams& p, int blocks, cudaStream_t st);
size_t encode_scratch_per_warp(int format, int hash_bits, int chain_bits, uint64_t max_src_len);
int encode_resident_warps(int sm_count);
cudaError_t launch_size_order(const uint64_t* d_size, uint32_t n, uint32_t* d_hist64, uint32_t* d_order, cudaStream_t st);
// LZ00's per-byte LCG keystream over bytes [skip, min(len[i], cap[i])) of every stream, read at in + in_off[i] and written at
// out + out_off[i] (keystream.cu; in place: the same pointer and offsets twice); cap may be null
cudaError_t launch_lcg_xor(const uint8_t* in, const uint64_t* d_in_off, uint8_t* out, const uint64_t* d_out_off, const uint64_t* d_len,
                           const uint64_t* d_cap, const uint32_t* d_key, uint32_t skip, uint32_t n, cudaStream_t st);
cudaError_t launch_scan(const uint8_t* image, uint64_t len, uint8_t* match, int format, cudaStream_t st);
cudaError_t launch_is_match(const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len, uint8_t* match, uint32_t n,
                            int format, cudaStream_t st);
// GetDecompressedSize of every stream (decoded_size_one, one thread per stream), and the status fix-up of a size scan
// (size_scan_status over the statuses of a size-only decode); ismatch.cu
cudaError_t launch_decoded_size(const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len, uint64_t* size,
                                int32_t* status, uint32_t n, int format, int byte_order, cudaStream_t st);
cudaError_t launch_size_scan_status(int32_t* status, uint32_t n, cudaStream_t st);
// the hits of the window [*d_base, *d_base + items) of an image (IsMatch to the image's end, is_match_one): the first `keep`
// offsets relative to *d_base, ascending, into rel, the number of all of them into *d_count.  A cub::DeviceSelect::If (two
// kernels); temp == nullptr only sets *temp_bytes.  ismatch.cu
cudaError_t launch_window_hits(const uint8_t* image, uint64_t len, const uint64_t* d_base, uint32_t items, int format, uint32_t* rel,
                               uint32_t keep, uint32_t* d_count, void* temp, size_t* temp_bytes, cudaStream_t st);
#ifdef __CUDACC__
// per-device scratch of aurora_scan_decode_device (scan_decode.cu): the walk state, the round's per-hit arrays, the select's
// and the scan's temporary storage, and the slots the round's hits are decoded into
struct ScanScratch {
    DevBuf state, hits, temp, slots;
    void release() {
        state.release();
        hits.release();
        temp.release();
        slots.release();
    }
};
// the rounds of aurora_scan_decode_device on `st` (arguments checked by the caller); counts its kernel launches into *launches
cudaError_t scan_decode_rounds(int format, const aurora_codec_opts* opts, const uint8_t* d_image, uint64_t len, uint64_t begin,
                               uint64_t max_size, uint64_t max_found, uint64_t* d_start, uint64_t* d_consumed, uint64_t* d_out_len,
                               uint8_t* d_dst_base, uint64_t dst_bytes, uint64_t* d_dst_off, uint64_t* found, uint64_t* next,
                               ScanScratch& scr, unsigned int* ticket, int sm_count, cudaStream_t st, uint64_t* launches);
#endif

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------
// mbarrier + 1-D TMA bulk copy (global -> shared), the sm_90+/sm_100a async staging path.
// SASS: UBLKCP.S.G + SYNCS.ARRIVE.TRANS64 / SYNCS.PHASECHK (see /opt/skills/guides/B200_PROFILING.md).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {   // release.cta: orders the arriving thread's earlier writes
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    // suspend-time hint (ns): the thread sleeps in hardware until the phase completes or the hint expires, so a
    // waiting warp does not burn issue slots polling
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(1000000u)
        : "memory");
    return ok != 0;
}
// (Measured and rejected, round 1: __nanosleep back-off in this loop; the polls are a third of the issued instructions
// of the pipelined flag-LZ kernel, but the hand-off latency it adds costs more than the issue slots it frees.)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// bytes and both addresses must be multiples of 16
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ uint32_t bswap32(uint32_t v) { return __byte_perm(v, 0, 0x0123); }
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
#endif

}  // namespace aurora
