"""ctypes mirror of include/aurora_cuda.h (constants + blittable structs).  No logic here."""
import ctypes as C

ABI_VERSION = 1

# aurora_status
OK, END_OF_STREAM, INVALID_IDENTIFIER, SIZE_MISMATCH, DST_TOO_SMALL, INVALID_DATA, NOT_SUPPORTED, \
    INVALID_ARGUMENT, CUDA_ERROR = range(9)
STATUS_NAMES = ["OK", "END_OF_STREAM", "INVALID_IDENTIFIER", "SIZE_MISMATCH", "DST_TOO_SMALL",
                "INVALID_DATA", "NOT_SUPPORTED", "INVALID_ARGUMENT", "CUDA_ERROR"]

# aurora_format
FMT_YAZ0, FMT_YAZ1, FMT_YAY0, FMT_MIO0, FMT_LZ10, FMT_LZ11, FMT_LZSS, FMT_LZ4, FMT_LZ4_BLOCK, \
    FMT_LZ4_LEGACY, FMT_LZO, FMT_SNAPPY, FMT_SNAPPY_BLOCK, FMT_PRS = range(1, 15)
# wrapper formats (a header around one of the cores above; decode on host buffers and on the device, the other device
# entry points do not take them)
FMT_GCLZ, FMT_CXLZ, FMT_COMP, FMT_LZ_3DS, FMT_LZ77, FMT_LEVEL5, FMT_LZON, FMT_LEVEL5_LZSS = range(15, 23)
FMT_AKLZ, FMT_LZ01, FMT_FCMP, FMT_IECP, FMT_MDB4, FMT_LZSEGA, FMT_GCZ = range(23, 30)   # header + LZSS headerless
FMT_SDPC = 30   # "SDPC" + size + LZO headerless
FMT_ECD = 31    # "ECD" header + plain bytes + LZSS(0x400, 0x42, 3, 0x3BE), or stored
FMT_LZ00 = 32   # 64-byte header + LZSS (Lzss0) under a per-byte LCG keystream
WRAPPER_FORMATS = list(range(15, 33))
FMT_LZHUDSON = 33   # a core format: Yay0 tokens under 32-bit big-endian flag words
FMT_LZ40, FMT_LZ60 = 34, 35   # core formats: LZ11-like 2/3/4-byte tokens (LE, length in the low nibble), negated flag bytes
FMT_BLZ = 37                  # core format (own kernel): Nintendo BLZ, parsed and written backwards from the end of the stream
FMT_SMSR00 = 36               # core format: MIO0 tokens, 16-bit BE mask words interleaved with the codes, literals in their own section
FORMAT_NAMES = {FMT_YAZ0: "Yaz0", FMT_YAZ1: "Yaz1", FMT_YAY0: "Yay0", FMT_MIO0: "MIO0", FMT_LZ10: "LZ10",
                FMT_LZ11: "LZ11", FMT_LZSS: "LZSS", FMT_LZ4: "LZ4", FMT_LZ4_BLOCK: "LZ4Block",
                FMT_LZ4_LEGACY: "LZ4Legacy", FMT_LZO: "LZO", FMT_SNAPPY: "Snappy",
                FMT_SNAPPY_BLOCK: "SnappyBlock", FMT_PRS: "PRS", FMT_GCLZ: "GCLZ", FMT_CXLZ: "CXLZ", FMT_COMP: "COMP",
                FMT_LZ_3DS: "3DS-LZ", FMT_LZ77: "LZ77", FMT_LEVEL5: "Level5", FMT_LZON: "LZOn", FMT_LEVEL5_LZSS: "Level5LZSS",
                FMT_AKLZ: "AKLZ", FMT_LZ01: "LZ01", FMT_FCMP: "FCMP", FMT_IECP: "IECP", FMT_MDB4: "MDB4", FMT_LZSEGA: "LZSega",
                FMT_GCZ: "GCZ", FMT_SDPC: "SDPC", FMT_ECD: "ECD", FMT_LZ00: "LZ00", FMT_LZHUDSON: "LZHudson", FMT_LZ40: "LZ40", FMT_LZ60: "LZ60", FMT_SMSR00: "SMSR00", FMT_BLZ: "BLZ"}

ENDIAN_LITTLE, ENDIAN_BIG, ENDIAN_DEFAULT = 0, 1, 2


class LzProps(C.Structure):
    _fields_ = [("windows_bits", C.c_int32), ("length_bits", C.c_int32), ("min_length", C.c_int32),
                ("max_length", C.c_int32), ("max_distance", C.c_int32), ("min_distance", C.c_int32),
                ("windows_start", C.c_int32), ("reserved", C.c_int32)]


class CodecOpts(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("byte_order", C.c_int32), ("quality", C.c_int32),
                ("max_window_bits", C.c_int32), ("strategy", C.c_int32), ("vram_mode", C.c_int32),
                ("lzss", LzProps), ("lzss_initial_fill", C.c_int32), ("lz4_block_size", C.c_uint32),
                ("lz4_verify", C.c_int32), ("yaz0_alignment", C.c_uint32), ("balance", C.c_uint32),
                ("lz77_type", C.c_uint32), ("lz77_chunk_size", C.c_uint32), ("level5_type", C.c_uint32),
                ("lz00_key", C.c_uint32), ("ecd_plain_size", C.c_uint32)]


# opts.strategy, library-specific bits (include/aurora_cuda.h): which byte-identical GPU match finder encodes
STRATEGY_COMPATIBILITY = 1
STRATEGY_PARALLEL_FINDER = 0x10000
STRATEGY_SERIAL_FINDER = 0x20000


def make_opts(byte_order=ENDIAN_DEFAULT, quality=-1, max_window_bits=0, strategy=0, vram_mode=-1,
              lzss=None, lzss_initial_fill=0, lz4_block_size=0, lz4_verify=0, yaz0_alignment=0, balance=0,
              lz77_type=0, lz77_chunk_size=0, level5_type=0, lz00_key=0, ecd_plain_size=0):
    o = CodecOpts()
    o.struct_size = C.sizeof(CodecOpts)
    o.byte_order = byte_order
    o.quality = quality
    o.max_window_bits = max_window_bits
    o.strategy = strategy
    o.vram_mode = vram_mode
    if lzss is not None:
        o.lzss = lzss
    o.lzss_initial_fill = lzss_initial_fill
    o.lz4_block_size = lz4_block_size
    o.lz4_verify = lz4_verify
    o.yaz0_alignment = yaz0_alignment
    o.balance = balance
    o.lz77_type = lz77_type
    o.lz77_chunk_size = lz77_chunk_size
    o.level5_type = level5_type
    o.lz00_key = lz00_key
    o.ecd_plain_size = ecd_plain_size
    return o


def _ceil_log2(x):
    b = 0
    while (1 << b) < x:
        b += 1
    return b


def lz_props_window(windows_size, max_length, min_length=3, windows_start=0, min_distance=1):
    """LzProperties ctor A (LzProperties.cs:46-55)."""
    return LzProps(_ceil_log2(windows_size), _ceil_log2(max_length - min_length) & 0xFF, min_length,
                   max_length, windows_size, min_distance, windows_start, 0)


def lz_props_bits(distance_bits, length_bits, threshold=2):
    """LzProperties ctor B (LzProperties.cs:57-66)."""
    md = 1 << distance_bits
    return LzProps(distance_bits, length_bits, threshold + 1, (1 << length_bits) + threshold, md, 1,
                   md - (1 << length_bits) - threshold, 0)


u8p = C.POINTER(C.c_uint8)
u64p = C.POINTER(C.c_uint64)
i32p = C.POINTER(C.c_int32)
