"""Batch entry points over the C ABI: many independent blobs at once (the north-star's new API).

`BatchCodec` owns one aurora_ctx (one per process; one process per GPU under torchrun, or all visible
GPUs of the box when device_mask == 0).  Host-buffer calls go through aurora_*_batch (H2D + kernel + D2H
inside the call); device-resident calls take torch CUDA tensors and only launch.
"""
import ctypes as C

import numpy as np

from . import _abi, _lib


class AuroraError(RuntimeError):
    pass


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def pack(blobs, align=16):
    """Concatenate byte blobs at `align`-byte aligned offsets -> (base u8 array, off u64, len u64)."""
    n = len(blobs)
    ln = np.array([len(b) for b in blobs], dtype=np.uint64)
    padded = (ln + np.uint64(align - 1)) & ~np.uint64(align - 1)
    off = np.zeros(n, dtype=np.uint64)
    if n > 1:
        off[1:] = np.cumsum(padded[:-1])
    total = int(padded.sum()) if n else 0
    base = np.zeros(max(total, 16), dtype=np.uint8)
    for i, b in enumerate(blobs):
        if len(b):
            base[int(off[i]):int(off[i]) + len(b)] = np.frombuffer(bytes(b), dtype=np.uint8) if not isinstance(b, np.ndarray) else b
    return base, off, ln


def layout(caps, align=16):
    caps = np.asarray(caps, dtype=np.uint64)
    padded = (caps + np.uint64(align - 1)) & ~np.uint64(align - 1)
    off = np.zeros(len(caps), dtype=np.uint64)
    if len(caps) > 1:
        off[1:] = np.cumsum(padded[:-1])
    return caps, off, (int(padded.sum()) if len(caps) else 0)


class BatchCodec:
    def __init__(self, device_mask=0):
        self._L = _lib.load()
        self._ctx = self._L.aurora_init(device_mask)
        if not self._ctx:
            raise AuroraError("aurora_init failed: " + self._L.aurora_last_error_string(None).decode() +
                              " (this engine has no CPU fallback; a B200 is required)")

    def close(self):
        if self._ctx:
            self._L.aurora_shutdown(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def device_count(self):
        return self._L.aurora_ctx_device_count(self._ctx)

    @property
    def kernel_launches(self):
        return int(self._L.aurora_kernel_launch_count(self._ctx))

    def _check(self, rc, what):
        if rc != _abi.OK:
            raise AuroraError(f"{what}: {_abi.STATUS_NAMES[rc]}: {self._L.aurora_last_error_string(self._ctx).decode()}")

    # ------------------------------------------------------------------ host buffers (packed numpy arrays)
    def decode_packed(self, fmt, base, off, ln, dst, doff, caps, opts=None):
        opts = opts or _abi.make_opts()
        n = len(off)
        out_len = np.zeros(n, dtype=np.uint64)
        consumed = np.zeros(n, dtype=np.uint64)
        status = np.zeros(n, dtype=np.int32)
        rc = self._L.aurora_decode_batch(self._ctx, fmt, C.byref(opts), n, _ptr(base), _ptr(off), _ptr(ln), _ptr(dst),
                                         _ptr(doff), _ptr(caps), _ptr(out_len), _ptr(consumed), _ptr(status))
        self._check(rc, "aurora_decode_batch")
        return out_len, consumed, status

    def decode_batch(self, fmt, blobs, caps, opts=None):
        """-> (list of decoded bytes truncated to cap, out_len, consumed, status)"""
        base, off, ln = pack(blobs)
        caps, doff, total = layout(caps)
        dst = np.zeros(max(total, 16), dtype=np.uint8)
        out_len, consumed, status = self.decode_packed(fmt, base, off, ln, dst, doff, caps, opts)
        outs = [dst[int(doff[i]):int(doff[i]) + min(int(out_len[i]), int(caps[i]))].tobytes() for i in range(len(blobs))]
        return outs, out_len, consumed, status

    def decoded_size_packed(self, fmt, base, off, ln, opts=None, size_scan=False):
        """GetDecompressedSize of the streams base[off[i]:off[i] + ln[i]] -> (size u64, status i32)"""
        opts = opts or _abi.make_opts()
        n = len(off)
        out = np.zeros(n, dtype=np.uint64)
        status = np.zeros(n, dtype=np.int32)
        rc = self._L.aurora_decoded_size_batch(self._ctx, fmt, C.byref(opts), n, _ptr(base), _ptr(off), _ptr(ln),
                                               1 if size_scan else 0, _ptr(out), _ptr(status))
        self._check(rc, "aurora_decoded_size_batch")
        return out, status

    def decoded_size_batch(self, fmt, blobs, opts=None, size_scan=False):
        base, off, ln = pack(blobs)
        return self.decoded_size_packed(fmt, base, off, ln, opts, size_scan)

    def is_match_packed(self, fmt, base, off, ln, opts=None):
        """IsMatch of the streams base[off[i]:off[i] + ln[i]] -> bool array"""
        opts = opts or _abi.make_opts()
        n = len(off)
        m = np.zeros(n, dtype=np.uint8)
        rc = self._L.aurora_is_match_batch(self._ctx, fmt, C.byref(opts), n, _ptr(base), _ptr(off), _ptr(ln), _ptr(m))
        self._check(rc, "aurora_is_match_batch")
        return m.astype(bool)

    def is_match_batch(self, fmt, blobs, opts=None):
        base, off, ln = pack(blobs)
        return self.is_match_packed(fmt, base, off, ln, opts)

    def scan_offsets(self, fmt, image, opts=None):
        """IsMatch at every byte offset of `image` -> bool array (the data-parallel `-scan`)."""
        opts = opts or _abi.make_opts()
        a = np.frombuffer(bytes(image), dtype=np.uint8) if not isinstance(image, np.ndarray) else image
        m = np.zeros(max(len(a), 1), dtype=np.uint8)
        if len(a):
            rc = self._L.aurora_scan_offsets(self._ctx, fmt, C.byref(opts), _ptr(a), len(a), _ptr(m))
            self._check(rc, "aurora_scan_offsets")
        return m[:len(a)].astype(bool)

    def encode_bound(self, fmt, raw_len):
        return int(self._L.aurora_encode_bound(fmt, raw_len))

    def encode_packed(self, fmt, base, off, ln, dst, doff, caps, opts=None):
        opts = opts or _abi.make_opts()
        n = len(off)
        out_len = np.zeros(n, dtype=np.uint64)
        status = np.zeros(n, dtype=np.int32)
        rc = self._L.aurora_encode_batch(self._ctx, fmt, C.byref(opts), n, _ptr(base), _ptr(off), _ptr(ln), _ptr(dst),
                                         _ptr(doff), _ptr(caps), _ptr(out_len), _ptr(status))
        self._check(rc, "aurora_encode_batch")
        return out_len, status

    def encode_batch(self, fmt, blobs, opts=None):
        base, off, ln = pack(blobs)
        caps, doff, total = layout([self.encode_bound(fmt, len(b)) for b in blobs])
        dst = np.zeros(max(total, 16), dtype=np.uint8)
        out_len, status = self.encode_packed(fmt, base, off, ln, dst, doff, caps, opts)
        outs = [dst[int(doff[i]):int(doff[i]) + int(out_len[i])].tobytes() if status[i] == 0 else b"" for i in range(len(blobs))]
        return outs, status

    # ------------------------------------------------------------------ device-resident (torch CUDA tensors)
    def decode_device(self, fmt, d_src, d_off, d_len, d_dst, d_doff, d_cap, d_out_len, d_consumed, d_status,
                      opts=None, device=0, stream=None):
        """All arguments are torch CUDA tensors (uint8 / int64 / int32).  Asynchronous on `stream`.

        Every format aurora_decode_batch takes, the wrapper formats included (same results as decode_batch); an LZ77 call
        reads its chunk count back and an LZ00 call the total size of its keystream-free bodies, so both wait for `stream`.
        Source windows may repeat and overlap.  d_src must start 16-byte aligned."""
        opts = opts or _abi.make_opts()
        rc = self._L.aurora_decode_batch_device(
            self._ctx, device, fmt, C.byref(opts), d_off.numel(), d_src.data_ptr(), d_src.numel(), d_off.data_ptr(),
            d_len.data_ptr(), d_dst.data_ptr(), d_doff.data_ptr(), d_cap.data_ptr(), d_out_len.data_ptr(),
            d_consumed.data_ptr(), d_status.data_ptr(), stream)
        self._check(rc, "aurora_decode_batch_device")

    def encode_device(self, fmt, d_src, d_off, d_len, d_dst, d_doff, d_cap, d_out_len, d_status, opts=None, device=0,
                      stream=None):
        """All arguments are torch CUDA tensors (uint8 / int64 / int32).  Asynchronous on `stream`.

        Every format encode_batch takes except BLZ, the wrapper formats included (same statuses, lengths and bytes as
        encode_batch / encode_packed with the same capacities); LZ77 with lz77_type 0xF7 (ChunkLZ10) reads its chunk count
        back and so waits for `stream`.  The source is never modified."""
        opts = opts or _abi.make_opts()
        rc = self._L.aurora_encode_batch_device(
            self._ctx, device, fmt, C.byref(opts), d_off.numel(), d_src.data_ptr(), d_src.numel(), d_off.data_ptr(),
            d_len.data_ptr(), d_dst.data_ptr(), d_doff.data_ptr(), d_cap.data_ptr(), d_out_len.data_ptr(),
            d_status.data_ptr(), stream)
        self._check(rc, "aurora_encode_batch_device")

    def decoded_size_device(self, fmt, d_src, d_off, d_len, d_size, d_status, opts=None, size_scan=False, device=0, stream=None):
        """GetDecompressedSize of device streams into d_size (int64) / d_status (int32): the answers of decoded_size_batch.
        d_src must start 16-byte aligned.  Asynchronous on `stream` (a cudaStream_t handle; None = the library's stream)."""
        opts = opts or _abi.make_opts()
        rc = self._L.aurora_decoded_size_batch_device(
            self._ctx, device, fmt, C.byref(opts), d_off.numel(), d_src.data_ptr(), d_src.numel(), d_off.data_ptr(),
            d_len.data_ptr(), 1 if size_scan else 0, d_size.data_ptr(), d_status.data_ptr(), stream)
        self._check(rc, "aurora_decoded_size_batch_device")

    def is_match_device(self, fmt, d_src, d_off, d_len, d_match, opts=None, device=0, stream=None):
        """IsMatch of device streams into d_match (uint8 or bool, one byte per stream).  Asynchronous on `stream`."""
        opts = opts or _abi.make_opts()
        rc = self._L.aurora_is_match_batch_device(self._ctx, device, fmt, C.byref(opts), d_off.numel(), d_src.data_ptr(),
                                                  d_off.data_ptr(), d_len.data_ptr(), d_match.data_ptr(), stream)
        self._check(rc, "aurora_is_match_batch_device")

    def scan_offsets_device(self, fmt, d_image, d_match, opts=None, device=0, stream=None):
        """IsMatch at every byte offset of a device image into d_match (d_image.numel() bytes).  Asynchronous on `stream`."""
        opts = opts or _abi.make_opts()
        rc = self._L.aurora_scan_offsets_device(self._ctx, device, fmt, C.byref(opts), d_image.data_ptr(), d_image.numel(),
                                                d_match.data_ptr(), stream)
        self._check(rc, "aurora_scan_offsets_device")

    def scan_decode_device(self, fmt, d_image, opts=None, max_size=1 << 26, begin=0, device=0, stream=None):
        """The CLI's `-scan` on a device image: every stream the offset walk from `begin` finds (IsMatch at a position, decode
        there with capacity `max_size`, resume after the consumed bytes of an OK stream, else one byte on), decoded on the
        device.  -> (d_start, d_consumed, d_out_len, d_dst, d_dst_off) on the image's device: int64 descriptors in walk order
        and the decoded bytes packed at 16-byte aligned offsets.  d_image must start 16-byte aligned.

        Calls aurora_scan_decode_device until the walk reaches the end, with output pieces of at least max_size bytes, and
        concatenates the pieces.  Each call reads back from the device, so this returns when the work on `stream` is done."""
        import torch
        opts = opts or _abi.make_opts()
        dev = d_image.device
        if stream is None:
            stream = torch.cuda.current_stream(dev).cuda_stream
        if not stream:
            # handle 0, torch's legacy default stream, means the library's own stream to the C ABI: finish the work that
            # wrote the image first (each call returns after its own work, so its results are ready when it returns)
            torch.cuda.current_stream(dev).synchronize()
        ts = torch.cuda.ExternalStream(stream, device=dev)
        length = d_image.numel()
        entries = 1 << 16
        piece = (max(int(max_size), 1 << 26) + 15) & ~15
        found, nxt = C.c_uint64(0), C.c_uint64(0)
        parts, dsts, base, pos = [], [], 0, begin
        with torch.cuda.stream(ts):
            while True:
                d = [torch.empty(entries, dtype=torch.int64, device=dev) for _ in range(4)]   # start, consumed, out_len, dst_off
                d_dst = torch.empty(piece, dtype=torch.uint8, device=dev)
                rc = self._L.aurora_scan_decode_device(
                    self._ctx, device, fmt, C.byref(opts), d_image.data_ptr(), length, pos, max_size, entries, d[0].data_ptr(),
                    d[1].data_ptr(), d[2].data_ptr(), d_dst.data_ptr(), piece, d[3].data_ptr(), C.byref(found), C.byref(nxt),
                    stream)
                self._check(rc, "aurora_scan_decode_device")
                k = found.value
                if k:
                    used = (int(d[3][k - 1]) + int(d[2][k - 1]) + 15) & ~15
                    parts.append((d[0][:k], d[1][:k], d[2][:k], d[3][:k] + base))
                    dsts.append(d_dst[:used])
                    base += used
                if nxt.value >= length:
                    break
                if k == 0:
                    raise AuroraError(f"aurora_scan_decode_device: no progress at offset {nxt.value}")
                pos = nxt.value
            if not parts:
                e = torch.empty(0, dtype=torch.int64, device=dev)
                return e, e.clone(), e.clone(), torch.empty(0, dtype=torch.uint8, device=dev), e.clone()
            cat = [torch.cat([p[i] for p in parts]) for i in range(4)]
            return cat[0], cat[1], cat[2], torch.cat(dsts), cat[3]

    def decode_device_sized(self, fmt, d_src, d_off, d_len, opts=None, size_scan=True, max_size=1 << 30, device=0, stream=None):
        """Decode device streams whose decoded sizes the caller does not know.
        -> (d_dst, d_dst_off, d_cap, d_out_len, d_consumed, d_status), all on `stream` (None: torch's current stream).

        The sizes come from decoded_size_device (with a size scan for the byte-LZ formats when size_scan is set).  A stream
        gets the capacity its size names when that is OK and at most `max_size` bytes, else 0, so a forged header cannot
        make this allocate gigabytes: such a stream reports the status of a fixed destination that is too small.  The
        destination windows are packed at 16-byte aligned offsets.  The one host read is the total, to allocate d_dst.
        The wrapper formats have no device-side size query, so this raises for them: pass capacities to decode_device
        (for example from decoded_size_batch on the host)."""
        import torch
        if d_src.data_ptr() % 16:
            raise AuroraError("decode_device_sized: INVALID_ARGUMENT: d_src must start at a 16-byte aligned address "
                              f"(data_ptr() % 16 == {d_src.data_ptr() % 16}; a sliced view may be misaligned)")
        dev = d_src.device
        if stream is None:
            stream = torch.cuda.current_stream(dev).cuda_stream
        ts = torch.cuda.ExternalStream(stream, device=dev)
        n = d_off.numel()
        with torch.cuda.stream(ts):
            d_size = torch.empty(n, dtype=torch.int64, device=dev)
            d_sst = torch.empty(n, dtype=torch.int32, device=dev)
            d_out_len = torch.empty(n, dtype=torch.int64, device=dev)
            d_consumed = torch.empty(n, dtype=torch.int64, device=dev)
            d_status = torch.empty(n, dtype=torch.int32, device=dev)
            if n == 0:
                return torch.zeros(16, dtype=torch.uint8, device=dev), d_size, torch.empty_like(d_size), d_out_len, d_consumed, d_status
            self.decoded_size_device(fmt, d_src, d_off, d_len, d_size, d_sst, opts, size_scan, device, stream)
            d_cap = torch.where((d_sst == _abi.OK) & (d_size <= max_size), d_size, torch.zeros_like(d_size))
            padded = (d_cap + 15) & ~15
            ends = torch.cumsum(padded, 0)
            d_dst_off = ends - padded
            total = int(ends[-1])
            d_dst = torch.empty(max(total, 16), dtype=torch.uint8, device=dev)
            self.decode_device(fmt, d_src, d_off, d_len, d_dst, d_dst_off, d_cap, d_out_len, d_consumed, d_status, opts, device, stream)
        return d_dst, d_dst_off, d_cap, d_out_len, d_consumed, d_status


_DEFAULT = None


def default_codec():
    """Process-wide BatchCodec (all visible devices)."""
    global _DEFAULT
    if _DEFAULT is None:
        _DEFAULT = BatchCodec(0)
    return _DEFAULT
