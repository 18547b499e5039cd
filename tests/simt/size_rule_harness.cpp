// tests/simt/size_rule_harness.cpp — GetDecompressedSize of one stream as both aurora_decoded_size_batch and the device's
// decoded_size_kernel compute it (decoded_size_one in csrc/ismatch.cu, everything above its "// ---- kernel" line, cut out of
// the real file by tests/test_size_rule_simt.py), compiled for the CPU.  TEST INFRASTRUCTURE.
#include "common.cuh"
#include ISMATCH_DEVICE_INC   // leaves `namespace aurora {` open
}  // namespace aurora

extern "C" int simt_decoded_size_one(int format, int byte_order, const uint8_t* p, uint64_t len, uint64_t* size) {
    return aurora::decoded_size_one(format, byte_order, p, len, size);
}

extern "C" int simt_size_scan_status(int status) { return aurora::size_scan_status(status); }
