// tests/simt/ismatch_harness.cpp — the IsMatch and GetDecompressedSize rules of csrc/ismatch.cu (everything above its
// "// ---- kernel" line, cut out of the real file by tests/test_simt_kernels.py) compiled for the CPU, so that the rules the
// IsMatch and offset-scan kernels run are compared with the oracle without a GPU.  TEST INFRASTRUCTURE.
#include "common.cuh"
#include ISMATCH_DEVICE_INC   // leaves `namespace aurora {` open
}  // namespace aurora

extern "C" int simt_is_match_one(const uint8_t* p, uint64_t len, int format) { return aurora::is_match_one(p, len, format); }

extern "C" int simt_core_decoded_size(int format, int byte_order, const uint8_t* p, uint64_t len, uint64_t* size) {
    return aurora::core_decoded_size(format, byte_order, p, len, size);
}
