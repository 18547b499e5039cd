"""The offset walk of aurora_scan_decode_device: walk_round and walk_target in csrc/scan_decode.cu, compiled for the CPU from the
real file (everything above its "// ---- kernel" line) and driven through rounds as the device drives it, against the walk
restated in Python on random tables of hits and decode outcomes.  No GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from auroralib.compression_b200 import _abi as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIMT = os.path.join(ROOT, "tests", "simt")
CSRC = os.path.join(ROOT, "auroralib", "compression_b200", "csrc")
U64 = np.uint64


@pytest.fixture(scope="module")
def walk(tmp_path_factory):
    build = tmp_path_factory.mktemp("scan_walk")
    src = open(os.path.join(CSRC, "scan_decode.cu")).read()
    inc = build / "scan_walk.inc"
    inc.write_text(src[:src.index("// ---- kernel\n")])
    so = build / "libsimt_scan_walk.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", SIMT, "-I", CSRC,
                           f'-DAURORA_REAL_COMMON="{os.path.join(CSRC, "common.cuh")}"', f'-DSCAN_WALK_INC="{inc}"',
                           os.path.join(SIMT, "scan_walk_harness.cpp"), "-o", str(so)])
    lib = C.CDLL(str(so))
    lib.simt_scan_walk.restype = None
    lib.simt_scan_walk.argtypes = [C.c_uint64, C.c_uint64] + [C.c_void_p] * 5 + [C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint64,
                                                                                    C.c_uint64, C.c_uint64] + [C.c_void_p] * 7
    lib.simt_walk_target.restype = C.c_uint64
    lib.simt_walk_target.argtypes = [C.c_uint64, C.c_int32, C.c_uint64]
    return lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def run(lib, t, begin, window, keep, budget, max_found, dst_bytes):
    n = len(t["hit"])
    out = [np.zeros(max(n, 1), dtype=U64) for _ in range(4)]
    found, nxt, rounds = C.c_uint64(), C.c_uint64(), C.c_uint64()
    lib.simt_scan_walk(t["len"], begin, _p(t["hit"]), _p(t["status"]), _p(t["consumed"]), _p(t["out_len"]), _p(t["cap"]), n, window,
                       keep, budget, max_found, dst_bytes, *[_p(o) for o in out], C.byref(found), C.byref(nxt), C.byref(rounds))
    k = found.value
    return [tuple(int(o[i]) for o in out) for i in range(k)], nxt.value, rounds.value


def ref_walk(t, begin, max_found=1 << 62, dst_bytes=1 << 62):
    """The walk of the header, with the hit table standing in for the bitmap and the decodes at max_size."""
    at = {int(h): i for i, h in enumerate(t["hit"])}
    entries, pos, i, visited = [], 0, begin, []
    while i < t["len"]:
        visited.append(i)
        k = at.get(i)
        if k is not None and t["status"][k] == A.OK:
            ol, c = int(t["out_len"][k]), int(t["consumed"][k])
            if len(entries) >= max_found or pos + ol > dst_bytes:
                return entries, i, visited
            entries.append((i, c, ol, pos))
            pos += (ol + 15) & ~15
            i += max(c, 1)
        else:
            i += 1
    return entries, t["len"], visited


def table(rng, length, density, ok_rate):
    """Random hits of an image of `length` bytes with outcomes: consumed 0, 1, short, to and past the last hit, past len."""
    hit = np.nonzero(rng.random(length) < density)[0].astype(U64)
    n = len(hit)
    status = np.where(rng.random(n) < ok_rate, A.OK, rng.choice([A.END_OF_STREAM, A.INVALID_DATA, A.DST_TOO_SMALL], n)).astype(np.int32)
    kind = rng.integers(0, 6, n)
    consumed = np.empty(n, dtype=U64)
    for k in range(n):
        h = int(hit[k])
        consumed[k] = [0, 1, int(rng.integers(2, 40)), int(rng.integers(1, max(2, length - h + 1))),
                       int(hit[-1]) - h + int(rng.integers(0, 3)), length - h + int(rng.integers(0, 50))][kind[k]]
        consumed[k] = max(int(consumed[k]), 0)
    out_len = rng.integers(0, 300, n).astype(U64)
    cap = out_len + rng.integers(0, 40, n).astype(U64)
    return {"len": length, "hit": hit, "status": status, "consumed": consumed, "out_len": out_len, "cap": cap}


ROUNDS = [(1 << 30, 1 << 20, 1 << 40), (64, 1 << 20, 1 << 40), (1 << 30, 5, 1 << 40), (1 << 30, 1 << 20, 700), (37, 3, 500)]


def test_walk_target_is_the_successor_rule(walk):
    assert walk.simt_walk_target(100, A.OK, 0) == 101
    assert walk.simt_walk_target(100, A.OK, 1) == 101
    assert walk.simt_walk_target(100, A.OK, 57) == 157
    for st in (A.END_OF_STREAM, A.DST_TOO_SMALL, A.SIZE_MISMATCH, A.INVALID_DATA):
        assert walk.simt_walk_target(100, st, 57) == 101


@pytest.mark.parametrize("seed", range(12))
def test_walk_matches_the_restated_walk(walk, seed):
    rng = np.random.default_rng(9100 + seed)
    t = table(rng, int(rng.integers(1, 3000)), [0.01, 0.1, 0.5, 1.0][seed % 4], [0.1, 0.5, 0.9][seed % 3])
    want, want_next, visited = ref_walk(t, 0)
    assert want_next == t["len"]
    for window, keep, budget in ROUNDS:
        got, nxt, rounds = run(walk, t, 0, window, keep, budget, 1 << 62, 1 << 62)
        assert (got, nxt) == (want, want_next), (seed, window, keep, budget)
    # begin at every walk position gives the matching suffix of the walk (offsets rebased)
    for b in visited[::max(1, len(visited) // 60)] + [t["len"]]:
        ref, ref_next, _ = ref_walk(t, b)
        for window, keep, budget in ROUNDS[1:]:
            got, nxt, _ = run(walk, t, b, window, keep, budget, 1 << 62, 1 << 62)
            assert (got, nxt) == (ref, ref_next), (seed, b, window, keep, budget)
        tail = [e for e in want if e[0] >= b]
        assert [e[:3] for e in ref] == [e[:3] for e in tail], (seed, b)


@pytest.mark.parametrize("seed", range(6))
def test_truncation_at_max_found_and_dst_bytes(walk, seed):
    rng = np.random.default_rng(9200 + seed)
    t = table(rng, int(rng.integers(500, 3000)), 0.05, 0.7)
    full, _, _ = ref_walk(t, 0)
    for window, keep, budget in ROUNDS:
        for mf in (0, 1, 2, len(full) // 2, len(full), len(full) + 1):
            got, nxt, _ = run(walk, t, 0, window, keep, budget, mf, 1 << 62)
            want, want_next, _ = ref_walk(t, 0, max_found=mf)
            assert (got, nxt) == (want, want_next), (seed, mf)
        for k in range(min(len(full), 8)):
            end = full[k][3] + full[k][2]   # the bytes of entry k end here
            for db in (end - 1, end, end + 15) if end else (0,):
                got, nxt, _ = run(walk, t, 0, window, keep, budget, 1 << 62, db)
                want, want_next, _ = ref_walk(t, 0, dst_bytes=db)
                assert (got, nxt) == (want, want_next), (seed, k, db)
                if db == end - 1:
                    assert len(got) == k and nxt == full[k][0]
        # pieces cut by max_found = 1 concatenate to the whole walk
        pieces, pos = [], 0
        while pos < t["len"]:
            got, nxt, _ = run(walk, t, pos, window, keep, budget, 1, 1 << 62)
            pieces += [e[:3] for e in got]
            assert nxt > pos or (not got and nxt == t["len"])
            pos = nxt
        assert pieces == [e[:3] for e in full]


def test_no_hits_and_tiny_images(walk):
    for length in (1, 15, 16, 5000):
        t = {"len": length, "hit": np.zeros(0, dtype=U64), "status": np.zeros(0, dtype=np.int32), "consumed": np.zeros(0, dtype=U64),
             "out_len": np.zeros(0, dtype=U64), "cap": np.zeros(0, dtype=U64)}
        for window, keep, budget in ROUNDS:
            got, nxt, rounds = run(walk, t, 0, window, keep, budget, 1 << 62, 1 << 62)
            assert (got, nxt) == ([], length)
            assert rounds == -(-length // min(window, 1 << 62))
