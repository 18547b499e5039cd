"""GetDecompressedSize of one stream as the library computes it on the host (aurora_decoded_size_batch) and on the device
(decoded_size_kernel of aurora_decoded_size_batch_device): decoded_size_one in csrc/ismatch.cu, compiled for the CPU from the
real file (everything above its "// ---- kernel" line) and compared with the oracle.  No GPU."""
import ctypes as C
import os
import subprocess

import pytest

from auroralib.compression_b200 import _abi as A
from tests.util import ALL_FORMATS, SIZED_FORMATS, decoded_size_blobs, fmt_id

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIMT = os.path.join(ROOT, "tests", "simt")
CSRC = os.path.join(ROOT, "auroralib", "compression_b200", "csrc")
BYTE_LZ = [f for f in ALL_FORMATS if f not in SIZED_FORMATS]


@pytest.fixture(scope="module")
def size_rule(tmp_path_factory):
    build = tmp_path_factory.mktemp("size_rule")
    src = open(os.path.join(CSRC, "ismatch.cu")).read()
    inc = build / "ismatch_device.inc"
    inc.write_text(src[:src.index("// ---- kernel\n")])
    so = build / "libsimt_size_rule.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", SIMT, "-I", CSRC,
                           f'-DAURORA_REAL_COMMON="{os.path.join(CSRC, "common.cuh")}"', f'-DISMATCH_DEVICE_INC="{inc}"',
                           os.path.join(SIMT, "size_rule_harness.cpp"), "-o", str(so)])
    lib = C.CDLL(str(so))
    lib.simt_decoded_size_one.restype = C.c_int
    lib.simt_decoded_size_one.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    lib.simt_size_scan_status.restype = C.c_int
    lib.simt_size_scan_status.argtypes = [C.c_int]
    return lib


def test_byte_lz_list_is_the_one_without_a_size_header():
    assert sorted(BYTE_LZ) == sorted([A.FMT_LZ4, A.FMT_LZ4_BLOCK, A.FMT_LZ4_LEGACY, A.FMT_LZO, A.FMT_SNAPPY, A.FMT_SNAPPY_BLOCK, A.FMT_PRS])


@pytest.mark.parametrize("fmt", ALL_FORMATS, ids=fmt_id)
def test_decoded_size_one_against_the_oracle(size_rule, oracle, fmt):
    blobs = decoded_size_blobs(oracle, fmt)
    for order in (A.ENDIAN_DEFAULT, A.ENDIAN_LITTLE, A.ENDIAN_BIG):
        opts = A.make_opts(byte_order=order)
        for b in blobs:
            size = C.c_uint64(77)
            st = size_rule.simt_decoded_size_one(fmt, order, b, len(b), C.byref(size))
            if fmt in BYTE_LZ:
                assert (st, size.value) == (A.NOT_SUPPORTED, 0), (fmt_id(fmt), order, b[:16].hex())
                continue
            rs, rst = oracle.decoded_size(fmt, b, opts)
            assert (size.value, st) == (rs, rst) or (st != 0 and rst != 0), (fmt_id(fmt), order, b[:16].hex(), size.value, st, rs, rst)
            if st != A.OK:
                assert size.value == 0


def test_decoded_size_one_rejects_wrapper_and_unknown_ids(size_rule):
    blob = b"GCLZ" + bytes(range(60))
    for fmt in (A.FMT_GCLZ, A.FMT_LZ77, A.FMT_LZ00, 0, 99):
        size = C.c_uint64(77)
        assert size_rule.simt_decoded_size_one(fmt, A.ENDIAN_DEFAULT, blob, len(blob), C.byref(size)) == A.INVALID_ARGUMENT, fmt
        assert size.value == 0


def test_size_scan_status_maps_only_dst_too_small(size_rule):
    for st in range(9):
        assert size_rule.simt_size_scan_status(st) == (A.OK if st == A.DST_TOO_SMALL else st)
