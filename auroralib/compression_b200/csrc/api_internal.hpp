// api_internal.hpp — entry points shared between api.cu, wrappers.cu and ismatch.cu (not part of the C ABI).
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "../../../include/aurora_cuda.h"

namespace aurora {

// core batches (api.cu): the bodies of aurora_decode_batch / aurora_encode_batch for the 14 core formats.
// raw_size: nullptr, or per-stream decoded sizes of headerless LZ10 / LZ11 / LZSS bodies (DecompressHeaderless).
// xor_key: nullptr, or per-stream LZ00 keys: the keystream pass (keystream.cu) runs on the device copy of every source
// stream before it is decoded, resp. over bytes [xor_skip, out_len) of every encoded stream.
// exact: write only the bytes every stream produced to the host (several sub-batches share one destination).
int decode_core_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                      const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                      const uint64_t* dst_cap, const uint64_t* raw_size, uint64_t* out_len, uint64_t* consumed, int32_t* status,
                      const uint32_t* xor_key = nullptr, bool exact = false);
int encode_core_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                      const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                      const uint64_t* dst_cap, uint64_t* out_len, int32_t* status, const uint32_t* xor_key = nullptr,
                      uint32_t xor_skip = 0);

// IsMatch and GetDecompressedSize rules of the core formats (ismatch.cu), the one copy of each.
// is_match_one: 1 match, 0 no match, -1 no rule for this format.  It also runs in the IsMatch and offset-scan kernels.
__host__ __device__ int is_match_one(const uint8_t* p, uint64_t len, int format);
// core_decoded_size: the header peek of BLZ and the flag-LZ formats.  A status; *size is 0 unless it is AURORA_OK.
// AURORA_INVALID_ARGUMENT for a format without a size header.
int core_decoded_size(int format, int byte_order, const uint8_t* p, uint64_t len, uint64_t* size);

// wrapper formats (wrappers.cu)
bool is_wrapper_format(int format);
int wrapped_decode_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                         const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                         const uint64_t* dst_cap, uint64_t* out_len, uint64_t* consumed, int32_t* status);
int wrapped_encode_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                         const uint64_t* src_off, const uint64_t* src_len, uint8_t* dst_base, const uint64_t* dst_off,
                         const uint64_t* dst_cap, uint64_t* out_len, int32_t* status);
int wrapped_decoded_size(int format, const uint8_t* p, uint64_t len, uint64_t* out_size);
int wrapped_is_match_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n, const uint8_t* src_base,
                           const uint64_t* src_off, const uint64_t* src_len, uint8_t* match);
uint64_t wrapped_encode_bound(int format, uint64_t raw_len, const aurora_codec_opts* opts);

}  // namespace aurora
