"""CPU tests of the host-side logic that needs no GPU: corpus generator determinism and class statistics, the
interface mirror's argument validation, and the N > 1 bookkeeping of bench.py under a 2-rank gloo group."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from auroralib.compression_b200 import _abi as A, corpus

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_corpus_is_deterministic_and_shaped():
    a, ca = corpus.generate_mix(20, 65536, seed=1)
    b, cb = corpus.generate_mix(20, 65536, seed=1)
    c, _ = corpus.generate_mix(20, 65536, seed=2)
    assert a.shape == (20, 65536) and a.dtype == torch.uint8 and torch.equal(a, b) and ca == cb and not torch.equal(a, c)
    assert "".join(ca[:10]) == corpus.CLASS_ORDER


def test_corpus_classes_compress_like_assets(oracle):
    """LZ10 ratios of the three C2 classes stay in the band the benchmark documents (DESIGN.md)."""
    for cls, lo, hi in (("T", 0.35, 0.60), ("M", 0.40, 0.70), ("X", 0.35, 0.60), ("B", 0.15, 0.60)):
        x = corpus.generate(cls, 8, 65536)
        comps, st = oracle.encode_batch(A.FMT_LZ10, [x[i].numpy().tobytes() for i in range(8)], A.make_opts(quality=8))
        ratio = sum(map(len, comps)) / (8 * 65536)
        assert (st == 0).all() and lo < ratio < hi, (cls, ratio)


def test_interface_mirror_validation():
    from auroralib.compression_b200 import CompressionSettings, LzProperties
    from auroralib.compression_b200.codecs import ArgumentException
    assert CompressionSettings().Quality == 8 and CompressionSettings.Maximum.Quality == 15
    with pytest.raises(ArgumentException):
        CompressionSettings(16)
    with pytest.raises(ArgumentException):
        CompressionSettings(8, 5)
    p = LzProperties.from_bits(12, 4, 2)
    assert (p.MinLength, p.MaxLength, p.MaxDistance, p.WindowsStart) == (3, 18, 4096, 4078)
    q = LzProperties(0x1000, 18, 3, 0xFEE)
    assert (q.WindowsBits, q.LengthBits, q.WindowsStart) == (12, 4, 0xFEE)


GLOO_WORKER = r'''
import os, sys, json
sys.path.insert(0, os.environ["AURORA_ROOT"])
import torch, torch.distributed as dist
from auroralib.compression_b200 import corpus
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
# the bench's N > 1 bookkeeping: per-rank shard seeds differ, the step time is the max over ranks, bytes add up
raw, cls = corpus.generate_mix(8, 4096, seed=0xA0120000 + 7919 * rank)
t = torch.tensor([10.0 + rank], dtype=torch.float64)
dist.all_reduce(t, op=dist.ReduceOp.MAX)
digest = torch.tensor([int(raw.sum())], dtype=torch.int64)
gathered = [torch.zeros(1, dtype=torch.int64) for _ in range(world)]
dist.all_gather(gathered, digest)
total = torch.tensor([raw.numel()], dtype=torch.int64)
dist.all_reduce(total)
if rank == 0:
    print(json.dumps({"tmax": t.item(), "digests": [int(g) for g in gathered], "total": int(total)}))
dist.barrier()
dist.destroy_process_group()
'''


def test_two_rank_gloo_bookkeeping(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER)
    env = dict(os.environ, AURORA_ROOT=ROOT, MASTER_ADDR="127.0.0.1")
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", "29617", str(script)], env=env, capture_output=True, text=True, timeout=240)
    assert out.returncode == 0, out.stderr[-2000:]
    import json
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    r = json.loads(line)
    assert r["tmax"] == 11.0 and r["total"] == 2 * 8 * 4096 and r["digests"][0] != r["digests"][1]


def test_reference_arm_ranks_other_than_zero_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         env=env, capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.parametrize("args", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "unused"]], ids=str)
def test_bench_rejects_arguments_it_cannot_honour(args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and out.stdout == "" and "error:" in out.stderr, out.stderr[-400:]


def test_bench_stream_mismatch_flags_exactly_the_windows_that_differ():
    """bench.stream_mismatch (the per-stream verifier of the C3 / C4 bench lines and of tests/test_baseline_sizes_gpu.py):
    ragged adjacent windows, an empty one, chunked over several passes."""
    import torch
    import bench
    g = torch.Generator().manual_seed(5)
    a = torch.randint(0, 256, (50000,), dtype=torch.uint8, generator=g)
    b = a.clone()
    ln = torch.tensor([100, 200, 0, 300, 50, 4096, 1, 7000], dtype=torch.int64)
    off = torch.cumsum(ln, 0) - ln + 7
    for i, at in ((1, 5), (4, 49), (7, 6999)):          # first, last and a middle byte of three windows
        b[int(off[i]) + at] ^= 0x5A
    b[int(off[3]) - 0 + 300 + 0] = b[int(off[3]) + 300]   # (untouched: the byte behind window 3 belongs to window 4)
    want = [False, True, False, False, True, False, False, True]
    for chunk in (1 << 30, 350, 64):
        assert bench.stream_mismatch(a, b, off, ln, chunk_bytes=chunk).tolist() == want


def test_bench_dump_batch_writes_the_reference_arm_sample(tmp_path, oracle):
    """`bench.py --dump-batch DIR` (the input of baseline/dotnet): packed.bin holds the LZ10 streams of the reference arm's
    sample at the offsets index.bin lists, and the oracle decodes them to 64 KiB each."""
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-batch", str(tmp_path), "--streams", "8"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-400:]
    idx = np.fromfile(tmp_path / "index.bin", dtype="<u8").reshape(-1, 3)
    packed = np.fromfile(tmp_path / "packed.bin", dtype=np.uint8)
    assert idx.shape == (8, 3) and (idx[:, 2] == 65536).all()
    for o, l, size in idx.tolist():
        blob = packed[o:o + l].tobytes()
        assert blob[0] == 0x10   # LZ10
        dec, out_len, consumed, st = oracle.decode(A.FMT_LZ10, blob, size)
        assert st == 0 and out_len == size and consumed == l
