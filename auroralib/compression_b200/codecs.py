"""Host-side mirror of the reference's operator interface for the hot path.

Each class keeps the names, argument meaning and error behaviour of its C# counterpart
(ICompressionAlgorithm = ICompressionDecoder + ICompressionEncoder, IProvidesDecompressedSize,
IEndianDependentFormat; /root/reference/src/AuroraLib.Compression/Interfaces/*.cs) and does its work
through the C ABI as a 1-element batch, exactly as the C# P/Invoke shim in csharp/ does.  Streams are
Python binary file objects (io.BytesIO, open(..., 'rb')): `source` is consumed from its current position
and left just past the consumed compressed bytes; `destination` receives the decoded bytes at its
current position (SURVEY.md §8b "Stream conventions").

There is no CPU implementation here: without libaurora_cuda.so and a B200 every call raises.
"""
import io

from . import _abi
from .batch import default_codec


# ---- exception taxonomy (SURVEY.md §8b "Error conventions") --------------------------------------
class EndOfStreamException(EOFError):
    pass


class InvalidIdentifierException(ValueError):
    pass


class DecompressedSizeException(ValueError):
    """Exceptions/DecompressedSizeException.cs:8-25"""

    def __init__(self, expected, actual):
        super().__init__(f"Expected {expected} bytes, but write {actual}bytes.")
        self.expected, self.actual = expected, actual


class InvalidDataException(ValueError):
    pass


class NotSupportedException(RuntimeError):
    pass


class ArgumentException(ValueError):
    pass


def _raise_for(status, expected=0, actual=0):
    if status == _abi.OK:
        return
    if status == _abi.END_OF_STREAM:
        raise EndOfStreamException()
    if status == _abi.INVALID_IDENTIFIER:
        raise InvalidIdentifierException()
    if status == _abi.SIZE_MISMATCH:
        raise DecompressedSizeException(expected, actual)
    if status == _abi.DST_TOO_SMALL:
        raise NotSupportedException("destination stream is not expandable")
    if status == _abi.INVALID_DATA:
        raise InvalidDataException()
    if status == _abi.NOT_SUPPORTED:
        raise NotSupportedException()
    if status == _abi.INVALID_ARGUMENT:
        raise ArgumentException()
    raise RuntimeError(f"aurora status {status}")


class Endian:
    Little = _abi.ENDIAN_LITTLE
    Big = _abi.ENDIAN_BIG


class CompressionSettings:
    """CompressionSettings.cs:38-50; default(CompressionSettings) is Quality 8 (:18-19)."""

    def __init__(self, quality=8, max_window_bits=0, strategy=0):
        if not 0 <= quality <= 15:
            raise ArgumentException("quality")
        if not (max_window_bits == 0 or 7 <= max_window_bits <= 28):
            raise ArgumentException("maxWindowBits")
        self.Quality, self.MaxWindowBits, self.Strategy = quality, max_window_bits, strategy


CompressionSettings.Fastest = CompressionSettings(0)
CompressionSettings.Fast = CompressionSettings(4)
CompressionSettings.Balanced = CompressionSettings(8)
CompressionSettings.High = CompressionSettings(12)
CompressionSettings.Maximum = CompressionSettings(15)


class LzProperties:
    """LzProperties.cs: ctor A (windowsSize, maxLength, minLength, windowsStart, minDistance) when the
    first argument is an int window size, ctor B (distanceBits, lengthBits, threshold) via from_bits."""

    def __init__(self, windows_size, max_length, min_length=3, windows_start=0, min_distance=1):
        self._p = _abi.lz_props_window(windows_size, max_length, min_length, windows_start, min_distance)

    @classmethod
    def from_bits(cls, distance_bits, length_bits, threshold=2):
        o = cls.__new__(cls)
        o._p = _abi.lz_props_bits(distance_bits, length_bits, threshold)
        return o

    WindowsBits = property(lambda s: s._p.windows_bits)
    LengthBits = property(lambda s: s._p.length_bits)
    MinLength = property(lambda s: s._p.min_length)
    MaxLength = property(lambda s: s._p.max_length)
    MaxDistance = property(lambda s: s._p.max_distance)
    MinDistance = property(lambda s: s._p.min_distance)
    WindowsStart = property(lambda s: s._p.windows_start)


def _remaining(stream):
    pos = stream.tell()
    data = stream.read()
    stream.seek(pos)
    return pos, data


class _Codec:
    """Shared plumbing: a 1-element batch through aurora_decode_batch / aurora_encode_batch."""
    FORMAT = 0
    Name = ""

    def _opts(self, settings=None):
        kw = {}
        if settings is not None:
            kw.update(quality=settings.Quality, max_window_bits=settings.MaxWindowBits, strategy=settings.Strategy)
        return _abi.make_opts(**kw)

    # IFormatInfoProvider.IsMatch
    def IsMatch(self, stream, fileNameAndExtension=None):
        _, data = _remaining(stream)
        return bool(default_codec().is_match_batch(self.FORMAT, [data], self._opts())[0])

    # ICompressionDecoder.Decompress(Stream source, Stream destination)
    def Decompress(self, source, destination=None):
        pos, data = _remaining(source)
        codec = default_codec()
        opts = self._opts()
        size, st = codec.decoded_size_batch(self.FORMAT, [data], opts, size_scan=True)
        if st[0] not in (_abi.OK,):
            # let the decoder produce the authoritative status (and the consumed position)
            size = [0]
        cap = self._capacity(int(size[0]), data)
        outs, out_len, consumed, status = codec.decode_batch(self.FORMAT, [data], [cap], opts)
        source.seek(pos + int(consumed[0]))
        ret = None
        if destination is None:
            destination = ret = io.BytesIO()
        destination.write(outs[0])
        _raise_for(int(status[0]), int(size[0]), int(out_len[0]))
        if ret is not None:
            ret.seek(0)
        return ret

    def _capacity(self, size, data):
        return size

    # ICompressionEncoder.Compress(ReadOnlySpan<byte> source, Stream destination, CompressionSettings settings)
    def Compress(self, source, destination=None, settings=None):
        outs, status = default_codec().encode_batch(self.FORMAT, [bytes(source)], self._opts(settings))
        _raise_for(int(status[0]))
        if destination is None:
            return io.BytesIO(outs[0])
        destination.write(outs[0])
        return None


class _SizedCodec(_Codec):
    # IProvidesDecompressedSize.GetDecompressedSize(Stream source): a peek
    def GetDecompressedSize(self, source):
        _, data = _remaining(source)
        # the whole remaining stream, as the reference does: MIO0 / Yay0 detect their byte order on the real stream length
        size, st = default_codec().decoded_size_batch(self.FORMAT, [data], self._opts())
        _raise_for(int(st[0]))
        return int(size[0])


class _EndianCodec:
    def __init__(self):
        self.FormatByteOrder = Endian.Big   # IEndianDependentFormat, class default Big


class Yaz0(_SizedCodec, _EndianCodec):
    """Nintendo/Yaz0.cs"""
    FORMAT, Name = _abi.FMT_YAZ0, "Nintendo Yaz0"

    def __init__(self):
        _EndianCodec.__init__(self)
        self.MemoryAlignment = 0

    def _opts(self, settings=None):
        o = super()._opts(settings)
        o.byte_order = self.FormatByteOrder
        o.yaz0_alignment = self.MemoryAlignment
        return o

    def _capacity(self, size, data):
        # Decompress retries with the byte-swapped size (Yaz0.cs:67-78): give the destination room for either
        swapped = int.from_bytes(size.to_bytes(4, "big"), "little")
        cands = [s for s in (size, swapped) if s <= 64 * max(len(data), 1) + 4096]
        return max(cands) if cands else size


class Yaz1(Yaz0):
    """Nintendo/Yaz1.cs"""
    FORMAT, Name = _abi.FMT_YAZ1, "Nintendo Yaz1"


class Yay0(_SizedCodec, _EndianCodec):
    """Nintendo/Yay0.cs"""
    FORMAT, Name = _abi.FMT_YAY0, "Nintendo Yay0"

    def __init__(self):
        _EndianCodec.__init__(self)
        self._explicit_order = False

    def _opts(self, settings=None):
        o = super()._opts(settings)
        # decode detects the order (DetectByteOrder<uint>(3)); FormatByteOrder only drives Compress
        o.byte_order = self.FormatByteOrder if (settings is not None or self._explicit_order) else _abi.ENDIAN_DEFAULT
        return o

    def Compress(self, source, destination=None, settings=None):
        return super().Compress(source, destination, settings or CompressionSettings())


class MIO0(Yay0):
    """Nintendo/MIO0.cs"""
    FORMAT, Name = _abi.FMT_MIO0, "Nintendo MIO0"


class LZ10(_SizedCodec):
    """Nintendo/LZ10.cs; GbaVramCompatibilityMode defaults to True (:33)"""
    FORMAT, Name = _abi.FMT_LZ10, "Nintendo LZ10"

    def __init__(self):
        self.GbaVramCompatibilityMode = True

    def _opts(self, settings=None):
        o = super()._opts(settings)
        o.vram_mode = 1 if self.GbaVramCompatibilityMode else 0
        return o


class LZ11(LZ10):
    """Nintendo/LZ11.cs; GbaVramCompatibilityMode defaults to False (:29)"""
    FORMAT, Name = _abi.FMT_LZ11, "Nintendo LZ11"

    def __init__(self):
        self.GbaVramCompatibilityMode = False


class LZSS(_SizedCodec):
    """Formats/Common/LZSS.cs; LZSS(LzProperties) with DefaultProperties ((byte)12, 4, 2)"""
    FORMAT, Name = _abi.FMT_LZSS, "Lempel-Ziv-Storer-Szymanski"

    def __init__(self, lz=None):
        self.LZ = lz or LzProperties.from_bits(12, 4, 2)

    def _opts(self, settings=None):
        o = super()._opts(settings)
        o.lzss = self.LZ._p
        return o


class LZ4(_Codec):
    """Formats/Common/LZ4.cs (+ LZ4.Frame.cs): FrameType / BlockSize / Flags; LZ4.HashAlgorithm as `Verify`"""
    FORMAT, Name = _abi.FMT_LZ4, "LZ4 Frame Compression"
    Legacy, LZ4FrameHeader = 0x184C2102, 0x184D2204

    def __init__(self):
        self.FrameType = LZ4.LZ4FrameHeader
        self.BlockSize = 0x400000
        self.Verify = False

    def _opts(self, settings=None):
        o = super()._opts(settings)
        o.lz4_block_size = self.BlockSize
        o.lz4_verify = 1 if self.Verify else 0
        return o

    def Compress(self, source, destination=None, settings=None):
        fmt = _abi.FMT_LZ4_LEGACY if self.FrameType == LZ4.Legacy else _abi.FMT_LZ4
        outs, status = default_codec().encode_batch(fmt, [bytes(source)], self._opts(settings))
        _raise_for(int(status[0]))
        if destination is None:
            return io.BytesIO(outs[0])
        destination.write(outs[0])
        return None


class LZ4Legacy(LZ4):
    """Formats/Common/LZ4Legacy.cs"""
    FORMAT, Name = _abi.FMT_LZ4_LEGACY, "LZ4 Legacy Compression"

    def __init__(self):
        super().__init__()
        self.FrameType = LZ4.Legacy


class LZO(_Codec):
    """Formats/Common/LZO.cs"""
    FORMAT, Name = _abi.FMT_LZO, "Lempel-Ziv-Oberhumer"


class Snappy(_Codec):
    """Formats/Common/Snappy.cs (framing format)"""
    FORMAT, Name = _abi.FMT_SNAPPY, "Snappy Frame"


class PRS(_Codec, _EndianCodec):
    """Sega/PRS.cs"""
    FORMAT, Name = _abi.FMT_PRS, "SEGA PRS"

    def __init__(self):
        _EndianCodec.__init__(self)

    def _opts(self, settings=None):
        o = super()._opts(settings)
        o.byte_order = self.FormatByteOrder
        return o


# ---- wrapper formats: a header around one of the cores above (AuroraLib.Compression.Nintendo; SURVEY.md 8f item 2) ----
class GCLZ(_SizedCodec):
    """Nintendo/GCLZ.cs: "GCLZ" + LZ10 (Pandora's Tower)"""
    FORMAT, Name = _abi.FMT_GCLZ, "GCLZ"


class CXLZ(_SizedCodec):
    """Sega/CXLZ.cs: "CXLZ" + LZ10"""
    FORMAT, Name = _abi.FMT_CXLZ, "CXLZ"


class COMP(_SizedCodec):
    """Sega/COMP.cs: "COMP" + LZ11"""
    FORMAT, Name = _abi.FMT_COMP, "COMP"


class LZ_3DS(_SizedCodec):
    """Nintendo/3DS-LZ.cs: "3DS-LZ\r\n" + LZ10"""
    FORMAT, Name = _abi.FMT_LZ_3DS, "3DS-LZ"


class LZ77(_SizedCodec):
    """Nintendo/LZ77.cs: "LZ77" + LZ10 / LZ11 / ChunkLZ10 (Type, ChunkSize :30-35)"""
    FORMAT, Name = _abi.FMT_LZ77, "Nintendo LZ77"
    LZ10_TYPE, LZ11_TYPE, CHUNK_LZ10_TYPE = 0x10, 0x11, 0xF7

    def __init__(self):
        self.Type = LZ77.LZ10_TYPE
        self.ChunkSize = 0x1000

    def _opts(self, settings=None):
        o = super()._opts(settings)
        o.lz77_type = self.Type
        o.lz77_chunk_size = self.ChunkSize
        return o


class Level5(_SizedCodec):
    """Level5/Level5.cs: u32 (type | size << 3) + OnlySave / LZ10 body (the Huffman, RLE and zlib types are not LZ codecs)"""
    FORMAT, Name = _abi.FMT_LEVEL5, "Level5 compression"
    ONLY_SAVE, LZ10_TYPE = 0, 1

    def __init__(self):
        self.Type = Level5.LZ10_TYPE

    def _opts(self, settings=None):
        o = super()._opts(settings)
        o.level5_type = self.Type
        return o

    def Compress(self, source, destination=None, settings=None):
        if settings is not None and settings.Quality == 0:
            self.Type = Level5.ONLY_SAVE   # Level5.cs:124-125 mutates the instance
        return super().Compress(source, destination, settings)

    def IsMatch(self, stream, fileNameAndExtension=None):
        raise NotSupportedException("Level5.IsMatch depends on zlib and the file extension (Level5.cs:35-50): not on the LZ hot path")


class LZOn(_SizedCodec):
    """Nintendo/LZOn.cs: "LZOn" header + LZO"""
    FORMAT, Name = _abi.FMT_LZON, "LZOn"


class Level5LZSS(_SizedCodec):
    """Level5/Level5LZSS.cs: "SSZL" header + LZSS with LZSS.Lzss0Properties"""
    FORMAT, Name = _abi.FMT_LEVEL5_LZSS, "Level5 lzss"


class _NoIdentifier:
    def IsMatch(self, stream, fileNameAndExtension=None):
        raise NotSupportedException(f"{type(self).__name__}.IsMatch is a heuristic on lengths / the file name, not an identifier: not on the LZ hot path")


class AKLZ(_SizedCodec):
    """Sega/AKLZ.cs: 12-byte identifier + BE size + LZSS body (DefaultProperties)"""
    FORMAT, Name = _abi.FMT_AKLZ, "AKLZ"


class LZ01(_SizedCodec):
    """Sega/LZ01.cs: "LZ01" + file length + size + 0 + LZSS body (Lzss0Properties)"""
    FORMAT, Name = _abi.FMT_LZ01, "LZ01"


class FCMP(_SizedCodec):
    """Extended/Marvelous/FCMP.cs: "FCMP" + size + constant + LZSS body (Lzss0Properties)"""
    FORMAT, Name = _abi.FMT_FCMP, "FCMP"


class IECP(_SizedCodec):
    """Extended/Marvelous/IECP.cs: "IECP" + size + LZSS body (Lzss0Properties)"""
    FORMAT, Name = _abi.FMT_IECP, "IECP"


class MDB4(_SizedCodec):
    """Extended/Specialized/MDB4.cs: 32-byte header + LZSS body (DefaultProperties)"""
    FORMAT, Name = _abi.FMT_MDB4, "MDB4"


class LZSega(_NoIdentifier, _SizedCodec):
    """Sega/LZSega.cs: compressed size + size + LZSS body (DefaultProperties)"""
    FORMAT, Name = _abi.FMT_LZSEGA, "LZSega"


class GCZ(_NoIdentifier, _SizedCodec):
    """Extended/Konami/GCZ.cs: size + LZSS body (Lzss0Properties)"""
    FORMAT, Name = _abi.FMT_GCZ, "Konami GCZ"


class SDPC(_SizedCodec):
    """Extended/Specialized/SDPC.cs: "SDPC" + size + LZO"""
    FORMAT, Name = _abi.FMT_SDPC, "SDPC"


class LZHudson(_SizedCodec):
    """HudsonSoft/LZHudson.cs: u32 BE size + Yay0 tokens under 4-byte big-endian flag words (a core format: the kernel decodes
    it directly, 32 tokens = one flag word per warp iteration).  IsMatch is the stream part of LZHudson.cs:31-32 (more than 8
    bytes, a non-zero first word); the reference also wants the ".lzHudson" extension when a file name is given."""
    FORMAT, Name = _abi.FMT_LZHUDSON, "LZHudson"


class BLZ(_SizedCodec):
    """Nintendo/BLZ.cs: parsed and written backwards from the footer at the end of the stream (its own kernel, decode_blz.cu)."""
    FORMAT, Name = _abi.FMT_BLZ, "Nintendo BLZ"


class SMSR00(_SizedCodec):
    """Nintendo/SMSR00.cs: "SMSR00" header, MIO0 tokens with 16-bit big-endian mask words interleaved with the codes and the
    literals in their own section (a core format)"""
    FORMAT, Name = _abi.FMT_SMSR00, "Nintendo SMSR00"


class LZ40(_SizedCodec):
    """Nintendo/LZ40.cs: 0x40 + u24 size, negated flag bytes, little-endian 2 / 3 / 4-byte match tokens (a core format)"""
    FORMAT, Name = _abi.FMT_LZ40, "Nintendo LZ40"

    def __init__(self):
        self.GbaVramCompatibilityMode = False   # LZ40.cs:35

    def _opts(self, settings=None):
        o = super()._opts(settings)
        o.vram_mode = 1 if self.GbaVramCompatibilityMode else 0
        return o


class LZ60(LZ40):
    """Nintendo/LZ60.cs: the LZ40 codec under identifier 0x60"""
    FORMAT, Name = _abi.FMT_LZ60, "Nintendo LZ60"


class ECD(_SizedCodec):
    """Extended/Specialized/ECD.cs: "ECD" + flag + plain size + compressed size + size (BE), PlainSize stored bytes + LZSS
    body with LzProperties(0x400, 0x42, 3, 0x3BE); quality 0, inputs of at most 16 bytes and incompressible inputs are stored"""
    FORMAT, Name = _abi.FMT_ECD, "ECD lzss"

    def __init__(self):
        self.PlainSize = 4   # ECD.cs:33

    def _opts(self, settings=None):
        o = super()._opts(settings)
        o.ecd_plain_size = self.PlainSize
        return o

    def _capacity(self, size, data):
        # GetDecompressedSize answers 0 when the compressed-size field does not fit the stream (ECD.cs:48-49); Decompress
        # does not look at that field, so the destination is sized by the header's size field (stored: by the payload)
        if len(data) >= 16:
            return max(size, int.from_bytes(data[12:16], "big"), len(data) - 16 if data[3] != 1 else 0)
        return size


class LZ00(_SizedCodec):
    """Sega/LZ00.cs: 64-byte header (file length, name, size, key) + LZSS body (Lzss0Properties) under a per-byte LCG
    keystream; the header's name field is always the reference's default "Temp.dat" """
    FORMAT, Name = _abi.FMT_LZ00, "LZ00"

    def Compress(self, source, destination=None, settings=None, key=None):
        # LZ00.cs:75-80: without a key the reference takes the Unix time of the call
        if key is None:
            import time
            key = int(time.time())
        o = self._opts(settings)
        o.lz00_key = key & 0xFFFFFFFF
        outs, status = default_codec().encode_batch(self.FORMAT, [bytes(source)], o)
        _raise_for(int(status[0]))
        if destination is None:
            return io.BytesIO(outs[0])
        destination.write(outs[0])
        return None


WRAPPERS = [GCLZ, CXLZ, COMP, LZ_3DS, LZ77, Level5, LZOn, Level5LZSS, AKLZ, LZ01, FCMP, IECP, MDB4, LZSega, GCZ, SDPC, ECD, LZ00]
ALGORITHMS = [Yaz0, Yaz1, Yay0, MIO0, LZ10, LZ11, LZSS, LZ4, LZ4Legacy, LZO, Snappy, PRS, LZHudson, LZ40, LZ60, SMSR00, BLZ] + WRAPPERS
