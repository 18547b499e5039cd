/*
 * aurora_cuda.h — C ABI of libaurora_cuda.so, the B200-native batched LZ-family codec engine.
 *
 * This is the drop-in boundary for the hot path of Venomalia/AuroraLib.Compression (managed C#):
 * every entry point below is what a P/Invoke (or ctypes / cgo / JNI) binding would call in place of
 * the reference's managed loops.  Plain pointers and sizes only; no CUDA or torch types.
 *
 * Reference interfaces replaced (paths relative to the reference tree, src/AuroraLib.Compression/...):
 *   ICompressionDecoder.Decompress(Stream, Stream)            Interfaces/ICompressionDecoder.cs:24
 *   ICompressionEncoder.Compress(ReadOnlySpan<byte>, Stream, CompressionSettings)
 *                                                             Interfaces/ICompressionEncoder.cs:19
 *   IProvidesDecompressedSize.GetDecompressedSize(Stream)     Interfaces/IProvidesDecompressedSize.cs:20
 *   IEndianDependentFormat.FormatByteOrder                    Interfaces/IEndianDependentFormat.cs:13
 *   IFormatInfoProvider.IsMatch(Stream, ReadOnlySpan<char>)   e.g. Nintendo/Yaz0.cs:41-47, LZ10.cs:36-41
 *   CompressionSettings(quality, maxWindowBits, strategy)     CompressionSettings.cs:38-50
 *   LzProperties                                              LzProperties.cs:46-66
 *   exceptions -> status codes                                Exceptions/DecompressedSizeException.cs:8-25
 *
 * The same symbols (prefix ora_ instead of aurora_, no context argument) are exported by the CPU
 * oracle in oracle/ so that tests can A/B the two libraries.
 */
#ifndef AURORA_CUDA_H
#define AURORA_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AURORA_ABI_VERSION 1

/* ---- per-stream status: 1:1 with the reference's exception taxonomy (SURVEY.md §8b) ---- */
typedef enum aurora_status {
    AURORA_OK                 = 0,
    AURORA_END_OF_STREAM      = 1, /* EndOfStreamException: truncated input                            */
    AURORA_INVALID_IDENTIFIER = 2, /* InvalidIdentifierException: wrong magic / type byte              */
    AURORA_SIZE_MISMATCH      = 3, /* DecompressedSizeException(expected, actual)                      */
    AURORA_DST_TOO_SMALL      = 4, /* NotSupportedException from a non-expandable destination stream   */
    AURORA_INVALID_DATA       = 5, /* InvalidDataException / ArgumentOutOfRangeException               */
    AURORA_NOT_SUPPORTED      = 6, /* NotSupportedException (LZ4 dictID, ...)                          */
    AURORA_INVALID_ARGUMENT   = 7, /* ArgumentException / ArgumentNullException                        */
    AURORA_CUDA_ERROR         = 8  /* the device failed; see aurora_last_error_string                  */
} aurora_status;

/* ---- formats on the hot path (SURVEY.md §8a D1-D11, E1-E6) ---- */
typedef enum aurora_format {
    AURORA_FMT_YAZ0         = 1,  /* Nintendo/Yaz0.cs                                        */
    AURORA_FMT_YAZ1         = 2,  /* Nintendo/Yaz1.cs (magic "Yaz1")                         */
    AURORA_FMT_YAY0         = 3,  /* Nintendo/Yay0.cs                                        */
    AURORA_FMT_MIO0         = 4,  /* Nintendo/MIO0.cs                                        */
    AURORA_FMT_LZ10         = 5,  /* Nintendo/LZ10.cs                                        */
    AURORA_FMT_LZ11         = 6,  /* Nintendo/LZ11.cs                                        */
    AURORA_FMT_LZSS         = 7,  /* Formats/Common/LZSS.cs (properties in opts.lzss)        */
    AURORA_FMT_LZ4          = 8,  /* LZ4.Decompress: legacy / v1 frame / skippable by magic  */
    AURORA_FMT_LZ4_BLOCK    = 9,  /* LZ4.DecompressBlockHeaderless / CompressBlockHeaderless */
    AURORA_FMT_LZ4_LEGACY   = 10, /* LZ4Legacy.cs (encode: legacy frame; decode == LZ4)      */
    AURORA_FMT_LZO          = 11, /* Formats/Common/LZO.cs (headerless LZO1X)                */
    AURORA_FMT_SNAPPY       = 12, /* Snappy.cs framing format                                */
    AURORA_FMT_SNAPPY_BLOCK = 13, /* Snappy.DecompressHeaderless / CompressHeaderless        */
    AURORA_FMT_PRS          = 14, /* Sega/PRS.cs                                             */
    /* wrapper formats: a header around one of the cores above (SURVEY.md 8f item 2; paths under
     * src/AuroraLib.Compression.Nintendo).  aurora_decode_batch resolves the headers on the host,
     * aurora_decode_batch_device on the device; the other device entry points do not take them. */
    AURORA_FMT_GCLZ         = 15, /* Nintendo/GCLZ.cs: "GCLZ" + LZ10                         */
    AURORA_FMT_CXLZ         = 16, /* Sega/CXLZ.cs: "CXLZ" + LZ10                             */
    AURORA_FMT_COMP         = 17, /* Sega/COMP.cs: "COMP" + LZ11                             */
    AURORA_FMT_LZ_3DS       = 18, /* Nintendo/3DS-LZ.cs: "3DS-LZ\r\n" + LZ10                 */
    AURORA_FMT_LZ77         = 19, /* Nintendo/LZ77.cs: "LZ77" + LZ10 / LZ11 / ChunkLZ10      */
    AURORA_FMT_LEVEL5       = 20, /* Level5/Level5.cs: u32 type|size<<3 + stored / LZ10 body */
    AURORA_FMT_LZON         = 21, /* Nintendo/LZOn.cs: "LZOn" header + LZO                   */
    AURORA_FMT_LEVEL5_LZSS  = 22, /* Level5/Level5LZSS.cs: "SSZL" header + LZSS (Lzss0)      */
    /* the LZSS-property family: a fixed header + LZSS.DecompressHeaderless with DefaultProperties or Lzss0Properties
     * (src/AuroraLib.Compression.Sega/Sega, src/AuroraLib.Compression-Extended) */
    AURORA_FMT_AKLZ         = 23, /* Sega/AKLZ.cs: 12-byte identifier + BE size, Default     */
    AURORA_FMT_LZ01         = 24, /* Sega/LZ01.cs: "LZ01" + length + size + 0, Lzss0         */
    AURORA_FMT_FCMP         = 25, /* Marvelous/FCMP.cs: "FCMP" + size + constant, Lzss0      */
    AURORA_FMT_IECP         = 26, /* Marvelous/IECP.cs: "IECP" + size, Lzss0                 */
    AURORA_FMT_MDB4         = 27, /* Specialized/MDB4.cs: 32-byte header, Default            */
    AURORA_FMT_LZSEGA       = 28, /* Sega/LZSega.cs: compressed size + size, Default         */
    AURORA_FMT_GCZ          = 29, /* Konami/GCZ.cs: size, Lzss0                              */
    AURORA_FMT_SDPC         = 30, /* -Extended/Specialized/SDPC.cs: "SDPC" + size + LZO      */
    AURORA_FMT_ECD          = 31, /* -Extended/Specialized/ECD.cs: "ECD" header + plain bytes + LZSS(0x400, 0x42, 3, 0x3BE) / stored */
    AURORA_FMT_LZ00         = 32, /* Sega/LZ00.cs: 64-byte header + LZSS (Lzss0) under a per-byte LCG keystream (on the device) */
    /* a core format (kernel path, device entry points included): Yay0 tokens under 32-bit big-endian flag words */
    AURORA_FMT_LZHUDSON     = 33, /* HudsonSoft/LZHudson.cs: u32 BE size + interleaved 4-byte flag words / tokens */
    AURORA_FMT_LZ40         = 34, /* Nintendo/LZ40.cs: 0x40 + u24 size; negated flag bytes, LE tokens of 2 / 3 / 4 bytes */
    AURORA_FMT_LZ60         = 35, /* Nintendo/LZ60.cs: the LZ40 codec under identifier 0x60                   */
    AURORA_FMT_SMSR00       = 36, /* Nintendo/SMSR00.cs: MIO0 tokens, 16-bit BE masks interleaved with the codes, literals in their own section */
    AURORA_FMT_BLZ          = 37  /* Nintendo/BLZ.cs: parsed and written backwards from the footer at the end of the stream (decode: own kernel;
                                     encode: reversal passes around the LZ10-layout encoder, host entry point only) */
} aurora_format;

typedef enum aurora_endian {
    AURORA_ENDIAN_LITTLE = 0,
    AURORA_ENDIAN_BIG    = 1,
    AURORA_ENDIAN_DEFAULT = 2 /* the class default: Big for Yaz0/Yay0/MIO0/PRS */
} aurora_endian;

/* LzProperties (LzProperties.cs:9-44).  Fill with aurora_lz_props_window / aurora_lz_props_bits. */
typedef struct aurora_lz_props {
    int32_t windows_bits;
    int32_t length_bits;
    int32_t min_length;
    int32_t max_length;
    int32_t max_distance;
    int32_t min_distance;
    int32_t windows_start;
    int32_t reserved;
} aurora_lz_props;

/* Blittable option block shared by decode and encode.  Zero-initialise, set struct_size. */
/* opts.strategy, library-specific bits: which of the two byte-identical match finders encodes the flag-byte formats
 * (LZ10 / BLZ, LZ11 / LZ40 / LZ60, Yaz0 / Yaz1, LZSS, MIO0, Yay0, LZHudson, SMSR00; every quality).  Default: the parallel one, except the
 * formats with matches longer than 32 bytes from quality 13 on, where the sequential replay is faster */
#define AURORA_STRATEGY_PARALLEL_FINDER 0x10000   /* one lane per window position, shared-memory tables (encode_lz_par.cu) */
#define AURORA_STRATEGY_SERIAL_FINDER   0x20000   /* sequential replay of LzChainMatchFinder (finder.cuh)                  */

typedef struct aurora_codec_opts {
    uint32_t struct_size;      /* sizeof(aurora_codec_opts)                                            */
    int32_t  byte_order;       /* aurora_endian: FormatByteOrder (Yaz0/Yay0/MIO0/PRS)                  */
    /* CompressionSettings (encode only).  quality < 0 means default(CompressionSettings) == 8.        */
    int32_t  quality;          /* 0..15                                                                */
    int32_t  max_window_bits;  /* 0 or 7..28                                                           */
    int32_t  strategy;         /* bit0 = CompresionStrategy.CompatibilityMode; bits 16 / 17 pick the GPU match finder
                                  (AURORA_STRATEGY_*_FINDER below) — the encoded bytes are the same either way      */
    int32_t  vram_mode;        /* LZ10/LZ11 GbaVramCompatibilityMode: -1 class default, 0 off, 1 on    */
    /* LZSS */
    aurora_lz_props lzss;      /* windows_bits == 0 -> LZSS.DefaultProperties ((byte)12, 4, 2)         */
    int32_t  lzss_initial_fill;/* LZSS.DecompressHeaderless initialFill                                */
    /* LZ4 (encode) */
    uint32_t lz4_block_size;   /* LZ4.BlockSize: 0 -> Block4MB                                         */
    int32_t  lz4_verify;       /* decode: 1 = verify XXH32 checksums (LZ4.HashAlgorithm set),
                                  0 = skip (HashAlgorithm == null, the library default)                */
    /* Yaz0 */
    uint32_t yaz0_alignment;   /* Yaz0.MemoryAlignment written by the encoder                          */
    uint32_t balance;          /* decode: hand streams to warps largest first (device counting sort by size class):
                                  0 = auto (host path: when max size > 2 x mean; device path: off), 1 = on, 2 = off */
    /* wrapper formats (encode) */
    uint32_t lz77_type;        /* LZ77.Type: 0 -> 0x10 (LZ10); 0x11 (LZ11); 0xF7 (ChunkLZ10)            */
    uint32_t lz77_chunk_size;  /* LZ77.ChunkSize: 0 -> 0x1000                                           */
    uint32_t level5_type;      /* Level5.Type: 0 -> 1 (LZ10); quality 0 always stores (OnlySave)        */
    uint32_t lz00_key;         /* LZ00 encode: the key written to the header (the reference uses the Unix time)  */
    uint32_t ecd_plain_size;   /* ECD.PlainSize (encode): 0 -> 4                                        */
} aurora_codec_opts;

typedef struct aurora_ctx aurora_ctx;

/* ---- lifetime ---- */
/* device_mask: bit i selects CUDA device i; 0 = all visible devices. */
aurora_ctx* aurora_init(uint32_t device_mask);
void        aurora_shutdown(aurora_ctx* ctx);
int         aurora_device_count(void);
int         aurora_ctx_device_count(const aurora_ctx* ctx);
int         aurora_abi_version(void);
const char* aurora_last_error_string(const aurora_ctx* ctx);
const char* aurora_status_string(int status);

/* pinned host memory for the blittable batch buffers (cudaHostAlloc) */
void* aurora_pinned_alloc(size_t bytes);
void  aurora_pinned_free(void* p);

/* LzProperties constructors (LzProperties.cs:46-55 and :57-66) */
void aurora_lz_props_window(aurora_lz_props* out, int32_t windows_size, int32_t max_length,
                            int32_t min_length, int32_t windows_start, int32_t min_distance);
void aurora_lz_props_bits(aurora_lz_props* out, int32_t distance_bits, int32_t length_bits,
                          int32_t threshold);
void aurora_codec_opts_init(aurora_codec_opts* opts);

/*
 * ---- batch entry points over HOST buffers (the call the C# shim makes) ----
 * Stream i occupies src_base[src_off[i] .. src_off[i]+src_len[i]).  Decoded bytes go to
 * dst_base[dst_off[i] .. dst_off[i]+dst_cap[i]).  All per-stream arrays have n entries.
 * Source windows may repeat and overlap (one file listed twice, several prefixes of one buffer, every scan hit of an image
 * read to its end): each stream's results are those it gets alone, and the source is never modified.  Destination windows
 * must not overlap.  This holds for every entry point below, the device-resident ones included.
 * Streams are sharded over the context's devices by size; no stream aborts the batch: errors
 * are reported in status[i].  Returns AURORA_OK, AURORA_INVALID_ARGUMENT or AURORA_CUDA_ERROR.
 * What the library writes into dst_base: the destination windows and nothing else, with ONE exception — windows that follow
 * each other in ascending order at most 15 bytes apart (the alignment padding of a packed batch) are copied back as one
 * piece, padding included, so those padding bytes are overwritten with unspecified values.  Offsets may have any alignment;
 * bytes in front of the first window, behind the last one and in gaps of 16 bytes or more are never touched.  (The wrapper
 * formats, which run several sub-batches over one destination, write only the bytes every stream produced.)
 */

/* IProvidesDecompressedSize.GetDecompressedSize for n streams.  Formats without a size header
 * (LZ4*, LZO, PRS) report AURORA_NOT_SUPPORTED unless size_scan != 0, in which case the stream
 * is parsed on the device without copying (a size-only pre-pass, SURVEY.md §7 "hard parts"). */
int aurora_decoded_size_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n,
                              const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len,
                              int size_scan, uint64_t* out_size, int32_t* status);

/* IsMatch(Stream) for n streams (magic checks and the LZ10/LZ11/PRS token-walk heuristics). */
int aurora_is_match_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n,
                          const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len,
                          uint8_t* match);

/* IsMatch at EVERY byte offset of one image: match[i] = IsMatch(image[i .. len)).  The data-parallel form of the CLI's
 * `-scan` loop (AuroraLib.Compression.CLI/Commands/ScanDecompressCommand.cs:23-39): the caller walks the bitmap, decodes
 * at the first hit and resumes after the consumed bytes.  `image` and `match` are host buffers of `len` bytes. */
int aurora_scan_offsets(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, const uint8_t* image, uint64_t len,
                        uint8_t* match);

/* Decompress(Stream source, Stream destination) for n streams.
 * out_len[i]  = bytes the reference would have written (may exceed dst_cap[i] on overshoot),
 * consumed[i] = source.Position after the call, relative to the start of stream i. */
int aurora_decode_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n,
                        const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len,
                        uint8_t* dst_base, const uint64_t* dst_off, const uint64_t* dst_cap,
                        uint64_t* out_len, uint64_t* consumed, int32_t* status);

/* Upper bound of the compressed size of a raw_len-byte input in `format` (all qualities). */
uint64_t aurora_encode_bound(int format, uint64_t raw_len);

/* Compress(ReadOnlySpan<byte> source, Stream destination, CompressionSettings) for n buffers. */
int aurora_encode_batch(aurora_ctx* ctx, int format, const aurora_codec_opts* opts, size_t n,
                        const uint8_t* src_base, const uint64_t* src_off, const uint64_t* src_len,
                        uint8_t* dst_base, const uint64_t* dst_off, const uint64_t* dst_cap,
                        uint64_t* out_len, int32_t* status);

/*
 * ---- device-resident variants (single device, inputs already in HBM; used by bench `value`) ----
 * All pointers are device pointers on `device` (an index into the context's device list);
 * descriptor arrays are device arrays too.  Decode / encode: src_off/dst_off must be multiples of 16.
 * `stream` is a cudaStream_t passed as void* (NULL = the context's own stream for that device);
 * the call is asynchronous with respect to the host: synchronise the stream before reading results.
 * Calls on ONE device must be stream-ordered with each other and with the host-buffer entry points: a device's work
 * counter, size-order array, encoder scratch and size-scan scratch (the zeroed destination offsets and the `consumed`
 * array of aurora_decoded_size_batch_device with size_scan != 0) are per device, not per call, so two batches of the same
 * device may not run concurrently (use one stream per device, or order the streams with events); different devices are
 * independent.
 * The wrapper formats (15-32) add per-device scratch of their own, shared by decode and encode: per-stream plans and
 * sub-stream (encode: core piece) descriptors and results, LZ77's chunk counts and their scan, and LZ00's keystream-free
 * bodies with their slot sizes and scan (decode).  A wrapped encode also uses the device's encoder scratch.
 * None of these calls synchronises with the host, reads a result on the host or copies the source to or from the host,
 * with four exceptions: aurora_decode_batch_device of LZ77 and of LZ00, aurora_encode_batch_device of LZ77 with
 * opts.lz77_type 0xF7, and aurora_scan_decode_device, which reads back once per round (below).
 *
 * aurora_decode_batch_device of the wrapper formats: out_len, consumed, status and the decoded bytes in
 * [dst_off[i], dst_off[i] + min(out_len[i], dst_cap[i])) are those aurora_decode_batch gives for the same streams, options
 * and capacities; nothing outside the destination windows is written, and the caller's source is never modified (LZ00's
 * keystream is lifted out of place, from the caller's bytes into one 16-byte aligned scratch slot per body, so bodies that
 * share source bytes are each decoded as if alone).  Same argument rules as the core formats
 * (16-byte aligned d_src_base, offsets multiples of 16); the sub-streams behind the headers start at any offset.  One
 * thread per stream resolves the header, the core kernels run on the sub-streams, one thread per stream merges the
 * results.  Kernel launches per call: 3 (header pass, core, merge) for GCLZ, CXLZ, COMP, 3DS-LZ, LZOn, SDPC, Level5LZSS and
 * the LZSS-property family; 4 for Level5 and ECD (+ a warp-per-stream copy of stored payloads / ECD's plain prefix); 7 for
 * LZ00 (header pass, the body slots' sizes, a two-kernel exclusive scan of them, the keystream pass into the slots, core,
 * merge); 9 for LZ77 (header pass, a two-kernel exclusive scan of the ChunkLZ10 chunk counts, chunk fill, LZ10 over stream
 * and chunk slots, LZ11 over the stream slots, redo selection, a redo LZ10 launch that decodes a file's failing chunk once
 * more so that its bytes win as in the reference's sequential loop, merge).  LZ77 READS ONE VALUE BACK: the batch's total
 * chunk count (a chunk table may be as long as its stream, so only the device knows how many descriptors the chunks need);
 * LZ00 READS ONE VALUE BACK too: the total size of the body slots (bodies may repeat or overlap in the source, so their
 * summed length is not bounded by src_total).  Either call returns after the stream has run its header pass and scan.
 * opts.balance is not applied
 * to the wrapper formats.  aurora_decoded_size_batch_device / aurora_is_match_batch_device / aurora_scan_offsets_device do
 * not take the wrapper formats: a wrapper caller passes its own capacities (e.g. from aurora_decoded_size_batch).
 */
int aurora_decode_batch_device(aurora_ctx* ctx, int device, int format, const aurora_codec_opts* opts,
                               size_t n, const uint8_t* d_src_base, uint64_t src_total,
                               const uint64_t* d_src_off, const uint64_t* d_src_len,
                               uint8_t* d_dst_base, const uint64_t* d_dst_off, const uint64_t* d_dst_cap,
                               uint64_t* d_out_len, uint64_t* d_consumed, int32_t* d_status,
                               void* stream);

/*
 * aurora_encode_batch_device: the core formats and the wrapper formats (15-32); BLZ answers AURORA_NOT_SUPPORTED (its reversal
 * passes and footer run only in aurora_encode_batch).  For the wrapper formats, out_len, status and the bytes
 * [dst_off[i], dst_off[i] + out_len[i]) of OK streams are those aurora_encode_batch gives for the same sources, options and
 * capacities, including its answers for a core piece without room (DST_TOO_SMALL, out_len 0), ChunkLZ10 end offsets past
 * 0xFFFF (INVALID_ARGUMENT), an lz77_type / level5_type without an encoder (NOT_SUPPORTED on every stream) and ECD's
 * ecd_plain_size above the source length (INVALID_ARGUMENT).  Nothing outside the destination windows is written and the
 * source is never modified (LZ00's keystream goes over the encoded output).  Same argument rules as the core formats.  One
 * thread per stream plans its core pieces (one piece, or one per ChunkLZ10 chunk in a worst-case slot), the unchanged core
 * encoder runs once over all pieces, and one warp per stream writes the header, the stored payloads and ECD's plain prefix,
 * moves bodies down in place (Level5 above 0xFFFFFF bytes, FCMP / IECP / LZSega / GCZ) and compacts the ChunkLZ10 chunks
 * behind their end-offset table.  Kernel launches per call: 3 (plan, core, finish); 4 for LZ00 (+ the keystream pass); 6 for
 * LZ77 with opts.lz77_type 0xF7 (plan, a two-kernel exclusive scan of the chunk counts, chunk fill, core, finish).  ChunkLZ10
 * READS ONE VALUE BACK, the batch's total chunk count, which sizes the piece descriptors: that call returns after the stream
 * has run its plan pass.  opts.balance is not applied to the wrapper formats.
 */
int aurora_encode_batch_device(aurora_ctx* ctx, int device, int format, const aurora_codec_opts* opts,
                               size_t n, const uint8_t* d_src_base, uint64_t src_total,
                               const uint64_t* d_src_off, const uint64_t* d_src_len,
                               uint8_t* d_dst_base, const uint64_t* d_dst_off, const uint64_t* d_dst_cap,
                               uint64_t* d_out_len, int32_t* d_status, void* stream);

/*
 * Device-resident GetDecompressedSize, IsMatch and offset scan: the same per-stream answers as aurora_decoded_size_batch,
 * aurora_is_match_batch and aurora_scan_offsets for every input, for the formats aurora_decode_batch_device takes (the core
 * formats and BLZ).  The wrapper formats, unknown ids and the formats the host entry point refuses return
 * AURORA_INVALID_ARGUMENT with a last error naming the host entry point, and launch nothing.  n == 0 / len == 0: AURORA_OK,
 * nothing launched.
 *
 * aurora_decoded_size_batch_device: d_out_size[i] / d_status[i] as aurora_decoded_size_batch with the same size_scan.  The
 * flag-LZ formats and BLZ are a header peek (one kernel); the byte-LZ formats (LZ4, LZ4 legacy, LZ4 block, LZO, Snappy,
 * Snappy block, PRS) report AURORA_NOT_SUPPORTED and size 0, unless size_scan != 0: then the decode kernel parses every
 * stream in size-only mode (no stores) and a second kernel turns its DST_TOO_SMALL into AURORA_OK; a failing stream keeps
 * its status and the length it reached.  d_src_base must be 16-byte aligned and, as for aurora_decode_batch_device, the
 * allocation readable up to the next multiple of 16 of src_total (the size scan stages its input with the same bulk copies).
 */
int aurora_decoded_size_batch_device(aurora_ctx* ctx, int device, int format, const aurora_codec_opts* opts, size_t n,
                                     const uint8_t* d_src_base, uint64_t src_total,
                                     const uint64_t* d_src_off, const uint64_t* d_src_len,
                                     int size_scan, uint64_t* d_out_size, int32_t* d_status, void* stream);

/* IsMatch of n device streams (one kernel, one thread per stream): d_match[i] as aurora_is_match_batch.  Any alignment;
 * only [d_src_off[i], d_src_off[i] + d_src_len[i]) is read.  LZ4 block and Snappy block have no IsMatch rule. */
int aurora_is_match_batch_device(aurora_ctx* ctx, int device, int format, const aurora_codec_opts* opts, size_t n,
                                 const uint8_t* d_src_base, const uint64_t* d_src_off, const uint64_t* d_src_len,
                                 uint8_t* d_match, void* stream);

/* IsMatch at every byte offset of a device image (one kernel): d_match[i] as aurora_scan_offsets.  Any alignment; len at
 * most 0xFFFFFFFF00.  The formats aurora_scan_offsets takes: the core formats except LZ4 block, Snappy block and BLZ. */
int aurora_scan_offsets_device(aurora_ctx* ctx, int device, int format, const aurora_codec_opts* opts,
                               const uint8_t* d_image, uint64_t len, uint8_t* d_match, void* stream);

/*
 * The CLI's `-scan` (ScanDecompressCommand.cs:23-39) on a device image: every stream the offset walk finds, decoded into device
 * memory.  For a format f, options opts, the image I of len bytes, a start `begin` and a capacity max_size, the walk W(begin) is
 *     i = begin
 *     while i < len:
 *         if aurora_scan_offsets(f, I)[i] and aurora_decode_batch(f, [I[i .. len)], cap = [max_size], opts) is AURORA_OK:
 *             emit (start = i, consumed, out_len, the out_len decoded bytes);  i += max(consumed, 1)
 *         else:
 *             i += 1
 * so a stream larger than max_size is not an entry (the decode reports DST_TOO_SMALL there and the walk steps by one byte).
 * Entries k = 0 .. *found - 1 of W(begin) are written in walk order to d_start[k], d_consumed[k], d_out_len[k] and the bytes
 * [d_dst_base + d_dst_off[k], + d_out_len[k]); d_dst_off[0] = 0 and d_dst_off[k + 1] = d_dst_off[k] + out_len[k] rounded up to
 * 16.  The call stops before the first entry that would be the max_found + 1-th or whose bytes would pass dst_bytes; *next is
 * that entry's start, or len when the walk reached the end, and W(*next) continues the walk exactly (no state between calls).
 * Formats: those aurora_scan_offsets takes (the core formats except LZ4 block, Snappy block and BLZ); the others are
 * AURORA_INVALID_ARGUMENT.  So are begin > len, max_size 0 or above 0xFFFFFFFF, len above 0xFFFFFFFF00, null pointers and a
 * d_image that is not 16-byte aligned; d_image must be readable up to len rounded up to 16, as d_src_base of
 * aurora_decode_batch_device.  len == 0 or begin == len: AURORA_OK, *found = 0, *next = len.  A rejected or empty call
 * launches nothing; so does a call with LZSS properties the decoder does not take (every decode reports AURORA_NOT_SUPPORTED, so
 * the walk has no entry: AURORA_OK, *found = 0, *next = len).  found and next are host pointers, the rest device memory on `device`.  Nothing is written outside the
 * entries' bytes and descriptors, and the image is never modified.
 * The walk runs in rounds from its position p.  Per round: the hits of a window [p, p + W) (a cub::DeviceSelect::If with the
 * IsMatch rule, 2 kernels; W adapts between 128 KiB and 1 GiB, at most 65 536 hits are kept), ONE HOST READ (the walk
 * position and the window's hit count), and when the window has hits: a capacity per hit (1 kernel; the byte-LZ formats first
 * run the decode kernel's size-only parse, +1 kernel, and turn its lengths into capacities, +1), slots for them by an
 * exclusive scan (2 kernels) cut at a budget of max(max_size, 256 MiB) decoded bytes (1), the decode kernel into the slots
 * (1), one warp that follows the walk and writes the descriptors (1), and a copy of the entries' bytes to d_dst_base (1):
 * 9 kernels per round (11 for the byte-LZ formats), 3 for a window without hits, plus a last window test that finds the
 * walk's end.  So THIS CALL READS BACK and returns after its work on `stream` is done (like LZ77 and LZ00 above).  Per-device
 * scratch: the walk state, the round's per-hit arrays (about 4 MiB), CUB's temporary storage, the slots (the budget), and the
 * device's work counter; the stream-ordering rule above applies.
 */
int aurora_scan_decode_device(aurora_ctx* ctx, int device, int format, const aurora_codec_opts* opts,
                              const uint8_t* d_image, uint64_t len, uint64_t begin, uint64_t max_size,
                              size_t max_found, uint64_t* d_start, uint64_t* d_consumed, uint64_t* d_out_len,
                              uint8_t* d_dst_base, uint64_t dst_bytes, uint64_t* d_dst_off,
                              uint64_t* found, uint64_t* next, void* stream);

/* Number of kernels this library has launched since aurora_init (all devices). */
uint64_t aurora_kernel_launch_count(const aurora_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* AURORA_CUDA_H */
