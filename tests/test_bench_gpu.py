"""bench.py on the GPU at a small size: --steps sets the timed decode launches, and --dump-outputs writes what the last of
them decoded, within the size limit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_decoded_streams(tmp_path):
    import torch
    import bench
    from auroralib.compression_b200 import corpus
    n = 300
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--streams", str(n), "--steps", "3", "--warmup", "0", "--no-configs",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 3 and line["gpu_launches"] == 3 and line["e2e"]["steps"] == 3
    files = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert sorted(files) == ["consumed", "decoded", "decoded_digest", "decoded_streams", "out_len", "status"]
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= bench.DUMP_BYTES
    assert (files["status"] == 0).all() and (files["out_len"] == bench.STREAM_BYTES).all() and files["consumed"].shape == (n,)
    assert (files["consumed"] > 0).all() and (files["consumed"] < bench.STREAM_BYTES + bench.STREAM_BYTES // 8 + 64).all()
    pick = files["decoded_streams"].astype(np.int64)
    assert len(pick) == bench.DUMP_STREAMS and len(set(pick.tolist())) == len(pick) and 0 <= pick.min() and pick.max() < n
    raw, _ = corpus.generate_mix(n, bench.STREAM_BYTES, seed=0xA0120000, device="cuda")
    assert np.array_equal(files["decoded"], raw[torch.as_tensor(pick, device=raw.device)].cpu().numpy().astype(np.float32))
    weights = np.arange(1, bench.STREAM_BYTES + 1, dtype=np.int64)
    assert np.array_equal(files["decoded_digest"], (raw.cpu().numpy().astype(np.int64) * weights).sum(1).astype(np.float64))
