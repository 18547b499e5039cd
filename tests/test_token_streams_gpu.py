"""The decode kernels on the B200, on streams written from each format's grammar by tests/tokens.py (see
tests/test_token_streams_simt.py for what the generators cover): about 2 000 generated streams per core format, some longer than
64 KiB, run valid and as truncated / short-capacity / larger-capacity variants.

  * the host entry point (aurora_decode_batch) with sources packed at 1-byte offsets and sentinel-filled gaps between the
    destination windows;
  * the device entry point (aurora_decode_batch_device) on torch tensors with a sentinel-filled destination;
  * once more through the host entry point with the largest-first hand-out (balance=1).

Every result must equal the oracle in status, out_len, consumed and (for a decoded stream) bytes, the two entry points must
equal each other in the same, and no byte outside the destination windows may change.  (Whole destination buffers are not
compared across the entry points: for the core formats the host entry point copies windows back whole, so bytes behind
out_len and the padding between windows less than 16 bytes apart are unspecified there, include/aurora_cuda.h.)"""
import functools

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from auroralib.compression_b200.batch import pack
from tests import tokens as T
from tests.test_token_streams_simt import options_key, variants
from tests.test_wrapped_device_gpu import _device_call, _device_inputs
from tests.util import fmt_id

pytestmark = pytest.mark.gpu

SENTINEL = 0xA5
PER_PROFILE = 280   # streams per (format, profile): 1 680-1 960 per format


@functools.lru_cache(maxsize=None)
def gpu_streams(fmt):
    from oracle import oracle as O
    rng = np.random.default_rng(104729 * fmt + 1)
    sizes = [300, 2000, 6000, 12000, 30000, 70000, 140000]
    out = []
    for p in T.profiles_of(fmt):
        for i in range(PER_PROFILE):
            out.append(T.generate(fmt, rng, p, size=int(rng.choice(sizes, p=[.2, .25, .2, .15, .1, .06, .04])), oracle=O))
    return out


def _cases(fmt):
    rng = np.random.default_rng(17 + fmt)
    ss = gpu_streams(fmt)
    cases = [(s, s.data, len(s.expect) if s.expect is not None else T.out_len([it for b in s.program for it in b])) for s in ss]
    cases += [(s, d, cap) for s in ss[::3] for d, cap in variants(rng, s)[1:]]
    groups = {}
    for c in cases:
        groups.setdefault(options_key(c[0]), []).append(c)
    return groups


def _check(fmt, what, datas, caps, ref, rlen, rcons, rst, dst, doff, olen, cons, st):
    bad = np.nonzero((st != rst) | (olen != rlen) | (cons != rcons))[0]
    if len(bad):
        i = int(bad[0])
        pytest.fail(f"{fmt_id(fmt)} {what}: {len(bad)}/{len(datas)} streams differ from the oracle; first #{i} ({len(datas[i])} bytes, "
                    f"cap {caps[i]}): status {st[i]} / {rst[i]}, out_len {olen[i]} / {rlen[i]}, consumed {cons[i]} / {rcons[i]}")
    for i in range(len(datas)):
        if rst[i] == 0:
            a = int(doff[i])
            if dst[a:a + len(ref[i])].tobytes() != ref[i]:
                pytest.fail(f"{fmt_id(fmt)} {what}: stream #{i} ({len(datas[i])} bytes, cap {caps[i]}) decodes to other bytes than the oracle")


def _host_gapped(codec, fmt, datas, caps, opts, rng):
    """1-byte packed sources; destination windows at odd offsets with sentinel gaps of 16-80 bytes and a margin"""
    base, off, ln = pack(datas, align=1)
    caps = np.asarray(caps, dtype=np.uint64)
    doff = np.zeros(len(datas), dtype=np.uint64)
    pos = 37
    for i in range(len(datas)):
        doff[i] = pos
        pos += int(caps[i]) + int(rng.integers(16, 80))
    dst = np.full(pos + 64, SENTINEL, dtype=np.uint8)
    olen, cons, st = codec.decode_packed(fmt, base, off, ln, dst, doff, caps, opts)
    covered = np.zeros(len(dst), dtype=bool)
    for i in range(len(datas)):
        covered[int(doff[i]):int(doff[i]) + int(caps[i])] = True
    outside = int((dst[~covered] != SENTINEL).sum())
    assert outside == 0, f"{fmt_id(fmt)}: the host path wrote {outside} bytes outside the destination windows"
    return dst, doff, olen, cons, st


@pytest.mark.parametrize("fmt", T.ALL, ids=fmt_id)
def test_token_streams_host_and_device(codec, oracle, fmt):
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(3 + fmt)
    total = 0
    for key, group in _cases(fmt).items():
        opts = group[0][0].opts
        datas, caps = [g[1] for g in group], [g[2] for g in group]
        ref, rlen, rcons, rst = oracle.decode_batch(fmt, datas, caps, opts)
        dst, doff, olen, cons, st = _host_gapped(codec, fmt, datas, caps, opts, rng)
        _check(fmt, f"host {key}", datas, caps, ref, rlen, rcons, rst, dst, doff, olen, cons, st)

        X = _device_inputs(datas, caps, dev, fill=SENTINEL)
        torch.cuda.synchronize(dev)
        _device_call(codec, fmt, X, opts)
        torch.cuda.synchronize(dev)
        d_dst = X["d_dst"].cpu().numpy()
        d_st, d_olen, d_cons = X["d_st"].cpu().numpy(), X["d_olen"].cpu().numpy().astype(np.uint64), X["d_cons"].cpu().numpy().astype(np.uint64)
        assert (d_st == st).all() and (d_olen == olen).all() and (d_cons == cons).all(), f"{fmt_id(fmt)} {key}: device and host results differ"
        _check(fmt, f"device {key}", datas, caps, ref, rlen, rcons, rst, d_dst, X["doff"], d_olen, d_cons, d_st)
        for i in np.nonzero(st == 0)[0]:
            a, b = int(doff[i]), int(X["doff"][i])
            assert dst[a:a + int(olen[i])].tobytes() == d_dst[b:b + int(olen[i])].tobytes(), f"{fmt_id(fmt)} {key}: stream #{i}"
        covered = np.zeros(len(d_dst), dtype=bool)
        for i in range(len(datas)):
            covered[int(X["doff"][i]):int(X["doff"][i]) + int(X["caps"][i])] = True
        outside = int((d_dst[~covered] != SENTINEL).sum())
        assert outside == 0, f"{fmt_id(fmt)}: the device path wrote {outside} bytes outside the destination windows"
        total += len(datas)
    assert total >= len(gpu_streams(fmt))
    print(f"{fmt_id(fmt)}: {len(gpu_streams(fmt))} generated streams, {total} decodes on each entry point, "
          f"{sum(len(s.expect or b'') > 65536 for s in gpu_streams(fmt))} longer than 64 KiB")


@pytest.mark.parametrize("fmt", [A.FMT_LZ10, A.FMT_LZ11, A.FMT_YAZ0, A.FMT_MIO0, A.FMT_LZ4_BLOCK, A.FMT_LZO, A.FMT_SNAPPY_BLOCK, A.FMT_PRS],
                         ids=fmt_id)
def test_token_streams_largest_first(codec, oracle, fmt):
    """balance=1: streams handed out largest first, on the same streams"""
    rng = np.random.default_rng(9 + fmt)
    for key, group in _cases(fmt).items():
        base_opts = group[0][0].opts
        opts = A.make_opts(byte_order=int(base_opts.byte_order), lzss=base_opts.lzss if fmt == A.FMT_LZSS else None,
                           lzss_initial_fill=int(base_opts.lzss_initial_fill), balance=1)
        datas, caps = [g[1] for g in group], [g[2] for g in group]
        ref, rlen, rcons, rst = oracle.decode_batch(fmt, datas, caps, base_opts)
        dst, doff, olen, cons, st = _host_gapped(codec, fmt, datas, caps, opts, rng)
        _check(fmt, f"balance=1 {key}", datas, caps, ref, rlen, rcons, rst, dst, doff, olen, cons, st)
