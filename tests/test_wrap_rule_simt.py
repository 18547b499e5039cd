"""The wrapper rules as the library runs them on the host (aurora_decode_batch) and on the device (the wrapper kernels of
aurora_decode_batch_device): wrap_resolve, wrap_chunk, wrap_merge and wrap_redo_chunk in csrc/wrappers.cu, compiled for the
CPU from the real file (everything above its "// ---- kernel" line) and compared with the oracle on valid, corrupt and
truncated streams of every wrapper format.  No GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A
from tests.test_wrappers import _opt_sets
from tests.util import corrupt, fmt_id, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIMT = os.path.join(ROOT, "tests", "simt")
CSRC = os.path.join(ROOT, "auroralib", "compression_b200", "csrc")
PARSE_HEADER = (1 << 64) - 1
MAX_SUB = 8192


@pytest.fixture(scope="module")
def wrap_rule(tmp_path_factory):
    build = tmp_path_factory.mktemp("wrap_rule")
    src = open(os.path.join(CSRC, "wrappers.cu")).read()
    inc = build / "wrappers_device.inc"
    inc.write_text(src[:src.index("// ---- kernel\n")])
    so = build / "libsimt_wrap_rule.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", SIMT, "-I", CSRC,
                           f'-DAURORA_REAL_COMMON="{os.path.join(CSRC, "common.cuh")}"', f'-DWRAPPERS_DEVICE_INC="{inc}"',
                           os.path.join(SIMT, "wrap_rule_harness.cpp"), "-o", str(so)])
    lib = C.CDLL(str(so))
    lib.simt_wrap_resolve.restype = C.c_int64
    lib.simt_wrap_resolve.argtypes = [C.c_int, C.c_char_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.simt_wrap_merge.restype = None
    lib.simt_wrap_merge.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.simt_wrap_redo_chunk.restype = C.c_int64
    lib.simt_wrap_redo_chunk.argtypes = [C.c_void_p, C.c_void_p]
    return lib


def resolve(lib, fmt, blob, cap):
    plan = np.zeros(10, dtype=np.uint64)
    subs = np.zeros(6 * MAX_SUB, dtype=np.uint64)
    k = lib.simt_wrap_resolve(fmt, blob, len(blob), cap, plan.ctypes.data, subs.ctypes.data, MAX_SUB)
    assert k >= 0
    return plan, subs[:6 * k].reshape(k, 6)


def merge(lib, fmt, plan, subs, r_out, r_cons, r_st):
    out = np.zeros(3, dtype=np.uint64)
    subs = np.ascontiguousarray(subs, dtype=np.uint64).reshape(-1)
    r_out, r_cons = np.asarray(r_out, dtype=np.uint64), np.asarray(r_cons, dtype=np.uint64)
    r_st = np.asarray(r_st, dtype=np.int32)
    lib.simt_wrap_merge(fmt, plan.ctypes.data, subs.ctypes.data if len(subs) else None, len(subs) // 6, r_out.ctypes.data,
                        r_cons.ctypes.data, r_st.ctypes.data, out.ctypes.data)
    return int(out[0]), int(out[1]), int(np.int64(out[2]))


def core_results(oracle, blob, cap, subs):
    """Each header-parsing sub-stream decoded by the oracle's core into its window of the stream's slot; None when a
    sub-stream is a headerless body (the oracle decodes those only inside its wrapper decode)."""
    r_out, r_cons, r_st, outs = [], [], [], []
    for core, off, ln, doff, raw, _ in subs.tolist():
        if raw != PARSE_HEADER:
            return None
        o, ol, cs, st = oracle.decode_batch(core, [blob[off:off + ln]], [max(0, cap - doff)])
        r_out.append(int(ol[0]))
        r_cons.append(int(cs[0]))
        r_st.append(int(st[0]))
        outs.append(o[0])
    return r_out, r_cons, r_st, outs


def streams(oracle, fmt, seed):
    """(blob, capacity, opts, raw or None) of valid, corrupt and truncated streams, with capacities 0, short, exact, larger"""
    rng = np.random.default_rng(seed)
    out = []
    for kw in _opt_sets(fmt):
        opts = A.make_opts(**({"quality": 8} | kw))
        raws = [synth(rng, int(n), i % 5) for i, n in enumerate([1, 7, 100, 1000, 4095, 4097, 9000, 20000])]
        comps, st = oracle.encode_batch(fmt, raws, opts)
        for i, (r, c) in enumerate(zip(raws, comps)):
            if st[i] != 0:
                continue
            out.append((c, len(r), opts, r))
            for cap in (0, max(0, len(r) - 17), len(r) + 100):
                out.append((c, cap, opts, None))
            for mode in range(5):
                out.append((corrupt(rng, c, mode), len(r) + int(rng.choice([0, 64])), opts, None))
    return out


@pytest.mark.parametrize("fmt", A.WRAPPER_FORMATS, ids=fmt_id)
def test_wrap_rules_against_the_oracle(wrap_rule, oracle, fmt):
    merged = 0
    for blob, cap, opts, raw in streams(oracle, fmt, 6100 + fmt):
        plan, subs = resolve(wrap_rule, fmt, blob, cap)
        _, rlen, rcons, rst = oracle.decode_batch(fmt, [blob], [cap], opts)
        want = (int(rlen[0]), int(rcons[0]), int(rst[0]))
        what = (fmt_id(fmt), len(blob), cap, blob[:16].hex())
        if plan[0] != A.OK or len(subs) == 0:
            # a header-level outcome: a header error or a stored payload, no core runs
            assert merge(wrap_rule, fmt, plan, subs, [0], [0], [0]) == want, what
            assert (int(plan[2]), int(plan[1]), int(plan[0])) == want, what
            continue
        if raw is not None:
            for core, off, ln, doff, rs, _ in subs.tolist():
                if rs == PARSE_HEADER:   # the core, run by the oracle at the sub-stream's doff, reproduces the raw bytes
                    o, _, _, st = oracle.decode_batch(core, [blob[off:off + ln]], [len(raw)])
                    assert st[0] == A.OK and raw[doff:doff + len(o[0])] == o[0], what
                else:                    # headerless: the raw size behind doff is the decoded size
                    assert rs + doff == oracle.decoded_size(fmt, blob, opts)[0] == len(raw), what
        res = core_results(oracle, blob, cap, subs)
        if res is None:
            continue
        r_out, r_cons, r_st, _ = res
        assert merge(wrap_rule, fmt, plan, subs, r_out, r_cons, r_st) == want, what
        merged += 1
    if fmt in (A.FMT_GCLZ, A.FMT_CXLZ, A.FMT_COMP, A.FMT_LZ_3DS, A.FMT_LZ77, A.FMT_LZON, A.FMT_SDPC):
        assert merged > 20


def test_lz77_chunk_table_and_redo(wrap_rule, oracle, bmp):
    """ChunkLZ10: the chunks wrap_chunk enumerates are the encoder's chunks at their decoded offsets; a cut file no longer ends
    where its table says (END_OF_STREAM from the header); a chunk whose last match overshoots (SIZE_MISMATCH, not the last
    chunk) is the one redone."""
    raw = bmp[:20000]
    c, st = oracle.encode(A.FMT_LZ77, raw, A.make_opts(quality=8, lz77_type=0xF7))
    assert st == 0
    plan, subs = resolve(wrap_rule, A.FMT_LZ77, c, len(raw))
    assert int(plan[5]) == len(subs) == 5 and int(plan[4]) == len(c)
    assert [int(s[3]) for s in subs] == [0x1000 * k for k in range(5)]
    cut = c[:len(c) - 40]
    plan_cut, _ = resolve(wrap_rule, A.FMT_LZ77, cut, len(raw))
    _, rlen, rcons, rst = oracle.decode_batch(A.FMT_LZ77, [cut], [len(raw)])
    assert (int(plan_cut[0]), int(plan_cut[1])) == (int(rst[0]), int(rcons[0])) == (A.END_OF_STREAM, len(cut))
    statuses = np.array([A.OK, A.SIZE_MISMATCH, A.OK, A.INVALID_DATA, A.OK], dtype=np.int32)
    assert wrap_rule.simt_wrap_redo_chunk(plan.ctypes.data, statuses.ctypes.data) == 1
    statuses = np.array([A.OK, A.OK, A.OK, A.OK, A.SIZE_MISMATCH], dtype=np.int32)   # the last chunk: nothing follows it
    assert wrap_rule.simt_wrap_redo_chunk(plan.ctypes.data, statuses.ctypes.data) == -1
    statuses = np.array([A.END_OF_STREAM, A.SIZE_MISMATCH, A.OK, A.OK, A.OK], dtype=np.int32)   # the first failure ends it
    assert wrap_rule.simt_wrap_redo_chunk(plan.ctypes.data, statuses.ctypes.data) == -1
