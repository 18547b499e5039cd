#!/usr/bin/env python
"""bench.py — the headline metric of BASELINE.json on its own configuration, plus the other configs of the metric.

metric   : batched LZ decode, decompressed GB/s out (LZ10 headline; Yaz0 / LZ4 ... under "configs"), and the fraction of
           the measured HBM roofline (compressed read + decompressed write bytes over the decode kernel's time)
headline : config C2 — 65 536 synthetic 64 KiB GBA/DS-style asset streams (classes T/M/X, 40/30/30 %), LZ10, encoded
           at quality 8 / VRAM mode on (the reference defaults) by this engine's GPU encoder (byte-identical to the
           oracle's, tests/test_encode_gpu.py); every decode is verified against the raw bytes
step     : one decode pass over the whole batch
value    : decompressed bytes / device time of the decode kernel with inputs already resident in HBM
e2e      : the same batch through aurora_decode_batch with pinned HOST buffers (H2D + kernel + D2H timed)
configs  : (N = 1 only) C3 Yaz0 / Yay0 / MIO0 (16 384 streams of 256 KiB - 4 MiB, half little-endian), C4 LZ4 / Snappy /
           LZO blocks (1 Mi streams of 4 - 64 KiB), C5 LZ10 / Yaz0 GPU encode of the C2 buffers — each with value,
           roofline and verified
N > 1    : ONE process (rank 0) drives all N devices through ONE library context (aurora_init over N devices): `value`
           = N x 65 536 streams decoded device-resident, one shard per device, launched back to back and timed with CUDA
           events per device (max over devices); `e2e` = ONE aurora_decode_batch call over all N x 65 536 host streams,
           cut and dealt to per-device worker threads by the library's scheduler (api.cu shard / for_each_shard) — the
           multi-GPU path of the north star.  Weak scaling, no collective on the data path; the other torchrun ranks
           only join the barriers.

`--impl reference` times the reference's CPU implementation of the same path — the C++ restatement in oracle/
(the reference is managed C# and there is no .NET runtime on the box; DESIGN.md "Oracle") — on all host threads.
"""
import argparse
import atexit
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "batched LZ10 decode throughput (decompressed GB/s out)"
UNIT = "GB/s"
STREAM_BYTES = 65536
FULL_STREAMS = 65536
QUALITY = 8
DUMP_BYTES = 64 * 10 ** 6      # --dump-outputs: size limit of all files together
DUMP_STREAMS = 192             # --dump-outputs: decoded streams kept whole (192 x 64 KiB as float32 = 48 MiB)
DUMP_SEED = 0xD0               # --dump-outputs: which streams, the same in every run and build


def workload_config(streams, n_gpus=1):
    return {
        "workload": "C2: LZ10 batched decode, 65536 synthetic 64 KiB GBA/DS-style asset streams per GPU",
        "format": "LZ10",
        "streams_per_gpu": streams,
        "stream_bytes": STREAM_BYTES,
        "classes": "T 40% / M 30% / X 30% (SURVEY.md 8d)",
        "encoder": "quality 8, GbaVramCompatibilityMode on (reference defaults)",
        "l2_policy": "inputs larger than L2 (compressed + decompressed working set >> 126 MB per step)",
        "multi_gpu": "single process, one library context over all devices; e2e = one aurora_decode_batch call sharded by the library" if n_gpus > 1 else "single device",
    }


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self.proc.kill)   # the sampler loops until stopped: it must not outlive a run that fails before stop()
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mxc = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx = mxc
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk)
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:
            sm = [float(l.split(",")[1]) for _, l in self.lines[-3:] if len(l.split(",")) > 2] or [0.0]
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def ncu_traffic(key, streams):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the decode kernel: NOT measured by this run — read from
    the committed `ncu --set full` capture of the same kernel and workload (profiles/ncu_traffic.json names the capture);
    null when the stream count differs or no capture of this build exists."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        e = d.get(key)
        if e and e.get("streams") == streams:
            return float(e["dram_bytes_per_launch"]), e.get("capture")
    except Exception:
        pass
    return None, None


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import numpy as np
    import torch
    from auroralib.compression_b200 import _abi as A, corpus
    from auroralib.compression_b200.batch import layout
    from oracle import oracle as O
    O.build()
    threads = O.hardware_threads()
    sample = min(args.streams, 8192)   # bounded sample of the C2 workload per step (512 MiB decoded)
    raw, _ = corpus.generate_mix(sample, STREAM_BYTES, device="cpu")
    raw_h = raw.numpy().reshape(-1)
    roff = np.arange(sample, dtype=np.uint64) * np.uint64(STREAM_BYTES)
    rlen = np.full(sample, STREAM_BYTES, dtype=np.uint64)
    caps, coff, ctotal = layout([STREAM_BYTES + STREAM_BYTES // 8 + 64] * sample)
    comp = np.zeros(ctotal + 16, dtype=np.uint8)
    clen, st = O.encode_packed(A.FMT_LZ10, raw_h, roff, rlen, comp, coff, caps, A.make_opts(quality=QUALITY), threads)
    assert (st == 0).all()
    if args.dump_batch:
        # the same sample for baseline/dotnet (the reference's C# decoder under Parallel.ForEach): packed.bin + index.bin
        os.makedirs(args.dump_batch, exist_ok=True)
        comp.tofile(os.path.join(args.dump_batch, "packed.bin"))
        np.stack([coff.astype(np.uint64), clen.astype(np.uint64), rlen], axis=1).astype("<u8").tofile(os.path.join(args.dump_batch, "index.bin"))
        print(json.dumps({"dumped": args.dump_batch, "streams": int(sample), "format": "LZ10"}), flush=True)
        return 0
    dst = np.zeros(sample * STREAM_BYTES + 16, dtype=np.uint8)
    times = []
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        out_len, consumed, status = O.decode_packed(A.FMT_LZ10, comp, coff, clen, dst, roff, rlen, None, threads)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    assert (status == 0).all() and np.array_equal(dst[:sample * STREAM_BYTES], raw_h)
    total = sum(times)
    value = sample * STREAM_BYTES * len(times) / total / 1e9
    sample_desc = f"{sample} of the {args.streams} C2 streams per step ({sample * STREAM_BYTES >> 20} MiB decoded), std::thread over {threads} host threads"
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(1000 * total / len(times), 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(args.streams, args.gpus),
        "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample_desc,
                         "note": "C++ restatement of the reference's managed decoder (no .NET runtime on the box)"},
        "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------ helpers (our arm)
def _i64(dev):
    import torch
    return dict(dtype=torch.int64, device=dev)


def pack_tight(c_buf, c_off, c_len, dev):
    """Compressed streams from their bound-sized slots to a tight, 16-byte aligned layout -> (packed, p_off, total)."""
    import torch
    n = c_len.numel()
    pad = (c_len + 15) & ~15
    p_off = torch.cumsum(pad, 0) - pad
    total = int(pad.sum())
    packed = torch.zeros(total + 16, dtype=torch.uint8, device=dev)
    slot = c_off[1:] - c_off[:-1] if n > 1 else None
    max_slot = int(slot.max()) if n > 1 else int(c_len.max())
    if max_slot <= (1 << 17):
        width = int(c_len.max())
        idx = torch.arange(width, device=dev).unsqueeze(0)
        step = max(1, (1 << 28) // max(width, 1))
        for s in range(0, n, step):
            e = min(n, s + step)
            mask = idx < c_len[s:e].unsqueeze(1)
            packed[(p_off[s:e].unsqueeze(1) + idx)[mask]] = c_buf[(c_off[s:e].unsqueeze(1) + idx)[mask]]
    else:
        co, po, cl = c_off.tolist(), p_off.tolist(), c_len.tolist()
        for i in range(n):
            packed[po[i]:po[i] + cl[i]] = c_buf[co[i]:co[i] + cl[i]]
    return packed, p_off, total


def gpu_encode(codec, fmt, raw, r_off, r_len, opts, dev, ts, device_index=0):
    """Encode on the GPU into bound-sized slots, pack tightly.  -> (packed, p_off, c_len, comp_total, encode_ms)"""
    import torch
    n = r_len.numel()
    lens = r_len.tolist()
    uniq = {}
    for v in set(lens):
        uniq[v] = (codec.encode_bound(fmt, v) + 15) & ~15
    bound = torch.tensor([uniq[v] for v in lens], **_i64(dev))
    c_off = torch.cumsum(bound, 0) - bound
    c_buf = torch.empty(int(bound.sum()) + 16, dtype=torch.uint8, device=dev)
    c_len = torch.zeros(n, **_i64(dev))
    e_st = torch.zeros(n, dtype=torch.int32, device=dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(ts):
        a.record(ts)
        codec.encode_device(fmt, raw, r_off, r_len, c_buf, c_off, bound, c_len, e_st, opts, device=device_index, stream=ts.cuda_stream)
        b.record(ts)
    ts.synchronize()
    assert int(e_st.abs().sum()) == 0, "GPU encode failed"
    packed, p_off, total = pack_tight(c_buf, c_off, c_len, dev)
    torch.cuda.synchronize(dev)   # the packing ran on torch's current stream, the decode launches go to `ts`
    del c_buf
    torch.cuda.empty_cache()
    return packed, p_off, c_len, total, a.elapsed_time(b)


def time_decode(codec, fmt, packed, p_off, c_len, d_dst, r_off, r_len, opts, steps, warmup, ts, device_index=0):
    """W warm-ups, K timed steps with CUDA events on the launching stream -> (avg kernel ms, total ms, status tensor)"""
    import torch
    dev = packed.device
    n = c_len.numel()
    d_olen, d_cons = torch.zeros(n, **_i64(dev)), torch.zeros(n, **_i64(dev))
    d_st = torch.zeros(n, dtype=torch.int32, device=dev)

    def once():
        codec.decode_device(fmt, packed, p_off, c_len, d_dst, r_off, r_len, d_olen, d_cons, d_st, opts, device=device_index, stream=ts.cuda_stream)

    for _ in range(warmup):
        once()
    ts.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with torch.cuda.stream(ts):
        for a, b in ev:
            a.record(ts)
            once()
            b.record(ts)
    ts.synchronize()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    return sum(step_ms) / len(step_ms), ev[0][0].elapsed_time(ev[-1][1]), d_st


def ragged_corpus(n, lo, hi, classes, seed, dev, group, odd=False):
    """n streams, decoded size log-uniform in [lo, hi], stream class round-robin over `classes` in groups; sorted by size
    (the library hands them out largest first).  -> (flat raw uint8, r_off, r_len, class letters per group)"""
    import torch
    from auroralib.compression_b200 import corpus
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    u = torch.rand(n, generator=g, dtype=torch.float64)
    sizes = torch.exp(math.log(lo) + u * (math.log(hi) - math.log(lo))).round().to(torch.int64).clamp_(lo, hi)
    if odd:
        # odd sizes: a Yaz0 header read in the wrong byte order then always claims >= 16 MiB, so the default-order decode of a
        # little-endian file fails at once and takes the reference's swapped-size retry (a size with a zero low byte can
        # read as a smaller, plausible size in the other order — an ambiguity of the reference's heuristic, Yaz0.cs:67-78)
        sizes = (sizes | 1).clamp_(max=hi - 1 if hi % 2 == 0 else hi)
    sizes, _ = torch.sort(sizes)
    r_len = sizes.to(dev)
    r_off = torch.cumsum(r_len, 0) - r_len
    raw = torch.empty(int(r_len.sum()) + 16, dtype=torch.uint8, device=dev)
    for gi, s in enumerate(range(0, n, group)):
        e = min(n, s + group)
        cls = classes[gi % len(classes)]
        width = int(sizes[e - 1])
        rows = corpus.generate(cls, e - s, width, seed + 7919 * gi, dev)
        if width <= (1 << 17):
            idx = torch.arange(width, device=dev).unsqueeze(0)
            mask = idx < r_len[s:e].unsqueeze(1)
            raw[(r_off[s:e].unsqueeze(1) + idx)[mask]] = rows[mask]
        else:
            ro, rl = r_off[s:e].tolist(), r_len[s:e].tolist()
            for i in range(e - s):
                raw[ro[i]:ro[i] + rl[i]] = rows[i, :rl[i]]
        del rows
    return raw, r_off, r_len


def stream_mismatch(a, b, off, ln, chunk_bytes=1 << 30):
    """Per-stream comparison of the windows [off, off + ln) of two flat uint8 tensors (windows ascending and disjoint)
    -> bool tensor, True where a window differs."""
    import torch
    n = ln.numel()
    out = torch.zeros(n, dtype=torch.bool, device=a.device)
    ends = (off + ln).tolist()
    offs = off.tolist()
    s = 0
    while s < n:
        e = s + 1
        while e < n and ends[e] - offs[s] <= chunk_bytes:
            e += 1
        lo, hi = offs[s], ends[e - 1]
        c = torch.cumsum((a[lo:hi] != b[lo:hi]).to(torch.int32), 0)
        c = torch.cat([torch.zeros(1, dtype=c.dtype, device=c.device), c])
        o, l = off[s:e] - lo, ln[s:e]
        out[s:e] = (c[o + l] - c[o]) != 0
        del c
        s = e
    return out


def dump_outputs(path, shards, n, size):
    """--dump-outputs: what the timed decode returned in its last step, as .npy files that two builds can be compared by.
    Per stream, over all devices' streams (device-major): status / out_len / consumed (float32 holds them exactly: 64 KiB
    streams) and decoded_digest, the sum of (position + 1) x byte over the stream's decoded bytes (exact in float64), which
    any change to one byte alters.  Besides, the decoded bytes of a seeded sample of whole streams (decoded_streams: their
    indices)."""
    import numpy as np
    import torch

    def digest(s):
        rows = s["d_dst"][:n * size].view(n, size)
        w = torch.arange(1, size + 1, dtype=torch.int64, device=s["dev"])
        return torch.cat([(rows[i:i + 1024].to(torch.int64) * w).sum(1) for i in range(0, n, 1024)]).cpu()

    per_stream = [torch.cat([s[k].cpu() for s in shards]).numpy().astype(np.float32) for k in ("st", "olen", "cons")]
    per_stream.append(torch.cat([digest(s) for s in shards]).numpy().astype(np.float64))
    total = len(shards) * n
    room = DUMP_BYTES - 4096 - sum(a.nbytes for a in per_stream)   # (4096: the .npy headers)
    rows = min(DUMP_STREAMS, total, room // (4 * size + 8))
    assert rows > 0, f"--dump-outputs: {total} streams do not fit {DUMP_BYTES} bytes"
    pick = np.sort(np.random.default_rng(DUMP_SEED).choice(total, size=rows, replace=False))
    decoded = torch.cat([s["d_dst"][:n * size].view(n, size)[torch.as_tensor(pick[pick // n == g] % n, device=s["dev"])].cpu()
                         for g, s in enumerate(shards)])
    os.makedirs(path, exist_ok=True)
    for name, a in zip(("status", "out_len", "consumed", "decoded_digest"), per_stream):
        np.save(os.path.join(path, name + ".npy"), a)
    np.save(os.path.join(path, "decoded_streams.npy"), pick.astype(np.float64))
    np.save(os.path.join(path, "decoded.npy"), decoded.numpy().astype(np.float32))


def bench_decode_config(codec, name, fmt, raw, r_off, r_len, dev, ts, peak, steps, warmup, orders, drop_unrepresentable=False,
                        enc_strategy=0):
    """Encode `raw` on the GPU, decode device-resident, verify.  `orders`: one entry per sub-batch of the streams — the byte
    order it is WRITTEN in (FormatByteOrder is a property of the encoding codec instance, so the two orders are two encode
    batches).  All streams are then decoded in ONE launch with the default byte order, as a reference user decodes a folder
    of mixed files with one codec instance: Yaz0 retries with the byte-swapped size (Yaz0.cs:67-78), Yay0 / MIO0 detect the
    order of every stream (DetectByteOrder); streams go to the warps largest first (opts.balance).
    drop_unrepresentable (LZO): the reference's LZO encoder writes two literal runs back to back when it shortens a match
    below MinLength (LZO.cs:168-188; tests/test_oracle_golden.py) and its own decoder does not round-trip such a stream;
    the streams that fail a first decode are left out of the timed batch and counted in `dropped_streams`."""
    import torch
    from auroralib.compression_b200 import _abi as A
    n = r_len.numel()
    d_dst = torch.zeros(raw.numel(), dtype=torch.uint8, device=dev)
    torch.cuda.synchronize(dev)
    enc_ms = 0.0
    dropped = 0
    cuts = [n * k // len(orders) for k in range(len(orders) + 1)]
    parts, base = [], 0
    for k, order in enumerate(orders):
        s, e = cuts[k], cuts[k + 1]
        packed_k, p_off_k, c_len_k, total_k, ms = gpu_encode(codec, fmt, raw, r_off[s:e].contiguous(), r_len[s:e].contiguous(),
                                                             A.make_opts(quality=QUALITY, byte_order=order, strategy=enc_strategy), dev, ts)
        enc_ms += ms
        parts.append((packed_k, p_off_k + base, c_len_k, total_k))
        base += (total_k + 15) & ~15
    if len(parts) == 1:
        packed, p_off, c_len = parts[0][0], parts[0][1], parts[0][2]
    else:
        packed = torch.zeros(base + 16, dtype=torch.uint8, device=dev)
        at = 0
        for pk, _, _, tk in parts:
            packed[at:at + tk] = pk[:tk]
            at += (tk + 15) & ~15
        p_off = torch.cat([q[1] for q in parts]).contiguous()
        c_len = torch.cat([q[2] for q in parts]).contiguous()
    del parts
    torch.cuda.empty_cache()
    torch.cuda.synchronize(dev)
    ro, rl = r_off.contiguous(), r_len.contiguous()
    dopts = A.make_opts(byte_order=A.ENDIAN_DEFAULT, balance=1)
    if drop_unrepresentable:
        _, _, d_st = time_decode(codec, fmt, packed, p_off, c_len, d_dst, ro, rl, dopts, 1, 0, ts)
        keep = (d_st == 0) & ~stream_mismatch(d_dst, raw, ro, rl)
        dropped = int((~keep).sum())
        d_dst.zero_()                                                 # the timed passes rewrite every kept window
        for i in (~keep).nonzero().flatten().tolist():                # the dropped ones are not part of the comparison below
            a, l = int(ro[i]), int(rl[i])
            d_dst[a:a + l] = raw[a:a + l]
        p_off, c_len, ro, rl = p_off[keep].contiguous(), c_len[keep].contiguous(), ro[keep].contiguous(), rl[keep].contiguous()
        torch.cuda.synchronize(dev)
    comp_bytes = int(c_len.sum())
    out_bytes = int(rl.sum())
    kernel_ms, _, d_st = time_decode(codec, fmt, packed, p_off, c_len, d_dst, ro, rl, dopts, steps, warmup, ts)
    ok = int(d_st.abs().sum()) == 0
    del packed
    torch.cuda.empty_cache()
    all_bytes = int(r_len.sum())
    ok = ok and bool(torch.equal(d_dst[:all_bytes], raw[:all_bytes])) and dropped * 100 < n
    achieved = (comp_bytes + out_bytes) / (kernel_ms * 1e-3) / 1e9
    res = {"format": name, "streams": n - dropped, "decoded_bytes": out_bytes, "compression_ratio": round(comp_bytes / out_bytes, 4),
           "value": round(out_bytes / (kernel_ms * 1e-3) / 1e9, 2), "unit": UNIT, "verified": ok, "launches_per_step": 1,
           "roofline": {"bound": "hbm", "achieved": round(achieved, 2), "frac": round(achieved / peak, 4),
                        "algorithmic_bytes": comp_bytes + out_bytes, "kernel_ms": round(kernel_ms, 4)},
           "gpu_encode_gbs_raw_in": round(all_bytes / (enc_ms * 1e-3) / 1e9, 2)}
    if drop_unrepresentable:
        res["dropped_streams"] = dropped
        res["dropped_reason"] = ("the reference's LZO encoder emits two literal runs back to back on these inputs (LZO.cs:168-188) and its "
                                 "own decoder does not round-trip them; decoder parity on them is covered by tests/test_baseline_sizes_gpu.py")
    del d_dst
    torch.cuda.empty_cache()
    return res


def other_configs(codec, dev, ts, peak, raw_c2, args):
    """C3, C4 and C5 of BASELINE.json (N = 1).  Every entry: value, roofline, verified."""
    import torch
    from auroralib.compression_b200 import _abi as A
    out = {}
    steps, warmup = 3, 2
    n2, size = raw_c2.shape
    # ---- C5: GPU encode of the C2 buffers (LZ10, Yaz0), verified by decoding on the GPU (the decoders are byte-exact
    #      against the oracle: tests/) and compared in size with the oracle's encoder on a sample
    r_off = torch.arange(n2, **_i64(dev)) * size
    r_len = torch.full((n2,), size, **_i64(dev))
    # (the two match finders write the same bytes: the search with one lane per window position — the kernel family BASELINE.json's
    #  north star names — is the default; the sequential replay of the reference's loop is timed next to it)
    def c5(name, fmt, strategy):
        opts = A.make_opts(quality=QUALITY, strategy=strategy)
        best, packed = 1e30, None
        for _ in range(2):
            if packed is not None:
                del packed
            packed, p_off, c_len, _, enc_ms = gpu_encode(codec, fmt, raw_c2.view(-1), r_off, r_len, opts, dev, ts)
            best = min(best, enc_ms)
        comp_bytes = int(c_len.sum())
        d_dst = torch.zeros(n2 * size + 16, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        _, _, d_st = time_decode(codec, fmt, packed, p_off, c_len, d_dst, r_off, r_len, opts, 1, 0, ts)
        ok = int(d_st.abs().sum()) == 0 and bool(torch.equal(d_dst[:n2 * size].view(n2, size), raw_c2))
        achieved = (n2 * size + comp_bytes) / (best * 1e-3) / 1e9
        out[name] = {"format": A.FORMAT_NAMES[fmt], "streams": n2, "raw_bytes": n2 * size, "quality": QUALITY,
                     "value": round(n2 * size / (best * 1e-3) / 1e9, 2), "unit": "GB/s raw in", "compression_ratio": round(comp_bytes / (n2 * size), 4),
                     "verified": ok, "roofline": {"bound": "hbm", "achieved": round(achieved, 2), "frac": round(achieved / peak, 4),
                                                  "algorithmic_bytes": n2 * size + comp_bytes, "kernel_ms": round(best, 3)}}
        del packed, d_dst
        torch.cuda.empty_cache()

    for name, fmt, strategy in (("C5_lz10_encode", A.FMT_LZ10, 0), ("C5_yaz0_encode", A.FMT_YAZ0, 0),
                                ("C5_lz10_encode_sequential_replay", A.FMT_LZ10, A.STRATEGY_SERIAL_FINDER),
                                ("C5_yaz0_encode_sequential_replay", A.FMT_YAZ0, A.STRATEGY_SERIAL_FINDER)):
        c5(name, fmt, strategy)
    # the other formats of the lane-per-position search (added at the end of round 2): reported, never allowed to break the line
    for name, fmt in (("C5_mio0_encode", A.FMT_MIO0), ("C5_yay0_encode", A.FMT_YAY0), ("C5_lz11_encode", A.FMT_LZ11)):
        try:
            c5(name, fmt, 0)
        except Exception as e:   # noqa: BLE001
            out[name] = {"format": A.FORMAT_NAMES[fmt], "error": f"{type(e).__name__}: {e}"[:200], "verified": False}
            import gc
            gc.collect()
            torch.cuda.empty_cache()
    if args.quick:
        return out
    # (the library's device buffers only grow — encoder scratch is sized by the largest stream of a batch — so every group of
    #  configs gets a context of its own and gives its memory back before the next one)
    from auroralib.compression_b200 import BatchCodec
    mask = 1 << dev.index
    # ---- C3: Yaz0 / Yay0 / MIO0, 16 384 streams of 256 KiB - 4 MiB (one third per format), half of each little-endian
    n3 = args.c3_streams // 3
    for k, (name, fmt) in enumerate((("C3_yaz0", A.FMT_YAZ0), ("C3_yay0", A.FMT_YAY0), ("C3_mio0", A.FMT_MIO0))):
        codec = BatchCodec(device_mask=mask)
        raw, r_off, r_len = ragged_corpus(n3, 256 << 10, 4 << 20, "TMXB", 0xA0130000 + k, dev, group=128, odd=True)
        out[name] = bench_decode_config(codec, A.FORMAT_NAMES[fmt], fmt, raw, r_off, r_len, dev, ts, peak, steps, warmup,
                                        orders=(A.ENDIAN_BIG, A.ENDIAN_LITTLE), enc_strategy=A.STRATEGY_SERIAL_FINDER)
        out[name]["sizes"] = ("log-uniform 256 KiB - 4 MiB, classes T/M/X/B; first half written big-endian, second half little-endian; decoded in one "
                              "launch with the default byte order (Yaz0: swapped-size retry, Yay0 / MIO0: per-stream order detection)")
        del raw
        codec.close()
        torch.cuda.empty_cache()
    # ---- C4: LZ4 / Snappy / LZO blocks, 1 Mi streams of 4 - 64 KiB
    raw, r_off, r_len = ragged_corpus(args.c4_streams, 4 << 10, 64 << 10, "TMX", 0xA0140000, dev, group=4096)
    for name, fmt in (("C4_lz4", A.FMT_LZ4_BLOCK), ("C4_snappy", A.FMT_SNAPPY_BLOCK), ("C4_lzo", A.FMT_LZO)):
        codec = BatchCodec(device_mask=mask)
        out[name] = bench_decode_config(codec, A.FORMAT_NAMES[fmt], fmt, raw, r_off, r_len, dev, ts, peak, steps, warmup, orders=(A.ENDIAN_DEFAULT,),
                                        drop_unrepresentable=fmt == A.FMT_LZO)
        out[name]["sizes"] = "log-uniform 4 - 64 KiB, classes T/M/X, raw blocks (capacity supplied by the caller)"
        codec.close()
    del raw
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from auroralib.compression_b200 import BatchCodec, _abi as A, corpus, _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev0 = torch.device("cuda", local_rank)
    cpu_group = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev0)
        # one NCCL collective up front (every rank joins the communicator); the barriers around the timed regions then run
        # on a gloo group: rank 0 drives EVERY device through one library context, and the NCCL barrier kernel of a waiting
        # rank would sit on that rank's GPU and time-slice with the decode kernels rank 0 launches there (measured: every
        # step took twice the kernel time at N = 2 and 4)
        t = torch.ones(1, device=dev0)
        dist.all_reduce(t)
        torch.cuda.synchronize()
        assert int(t.item()) == world
        cpu_group = dist.new_group(backend="gloo")

    def barrier():
        torch.cuda.set_device(dev0)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=cpu_group)
        torch.cuda.synchronize()

    if rank != 0:
        # the data path has no collective: rank 0 drives every device through one library context (see the docstring);
        # the other ranks only take part in the barriers around the timed regions
        for _ in range(4):
            barrier()
        dist.destroy_process_group()
        return 0

    G = max(1, min(world, torch.cuda.device_count()))
    codec = BatchCodec(device_mask=(1 << G) - 1 if world > 1 else 1 << local_rank)
    assert codec.device_count == G, f"library context holds {codec.device_count} of {G} devices"
    devs = [torch.device("cuda", i if world > 1 else local_rank) for i in range(G)]
    n, size = args.streams, STREAM_BYTES
    fmt = A.FMT_LZ10
    opts = A.make_opts(quality=QUALITY)
    peak, peak_src = measured_peak()

    # ---- per device: synthetic corpus, encoded by the engine's own GPU encoder (byte-identical to the oracle's)
    shards = []
    t_enc = 0.0
    for g, dev in enumerate(devs):
        torch.cuda.set_device(dev)
        ts = torch.cuda.Stream(device=dev)
        raw, classes = corpus.generate_mix(n, size, seed=0xA0120000 + 7919 * g, device=dev)
        r_off = torch.arange(n, **_i64(dev)) * size
        r_len = torch.full((n,), size, **_i64(dev))
        t0 = time.perf_counter()
        packed, p_off, c_len, comp_total, _ = gpu_encode(codec, fmt, raw.view(-1), r_off, r_len, opts, dev, ts, device_index=g)
        t_enc += time.perf_counter() - t0
        d_dst = torch.zeros(n * size + 16, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize(dev)
        shards.append(dict(dev=dev, ts=ts, raw=raw, classes=classes, r_off=r_off, r_len=r_len, packed=packed, p_off=p_off, c_len=c_len,
                           comp_total=comp_total, comp_bytes=int(c_len.sum()), d_dst=d_dst,
                           olen=torch.zeros(n, **_i64(dev)), cons=torch.zeros(n, **_i64(dev)), st=torch.zeros(n, dtype=torch.int32, device=dev)))
    out_bytes = n * size
    comp_bytes = sum(s["comp_bytes"] for s in shards)

    def decode_all():
        for g, s in enumerate(shards):
            codec.decode_device(fmt, s["packed"], s["p_off"], s["c_len"], s["d_dst"], s["r_off"], s["r_len"], s["olen"], s["cons"], s["st"],
                                device=g, stream=s["ts"].cuda_stream)

    def sync_all():
        for s in shards:
            s["ts"].synchronize()

    # ---- device-resident timing: W warm-ups, K timed steps, CUDA events on each device's launching stream
    warm = max(args.warmup, 3)
    for _ in range(warm):
        decode_all()
    sync_all()
    for s in shards:
        assert int(s["st"].abs().sum()) == 0 and torch.equal(s["d_dst"][:out_bytes].view(n, size), s["raw"]), "decode mismatch"
    sampler = ClockSampler(devs[0].index)
    sampler.start()
    time.sleep(0.25)
    barrier()
    launches0 = codec.kernel_launches
    evs = []
    for s in shards:
        torch.cuda.set_device(s["dev"])
        evs.append([(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)])
    t_wall0 = time.time()
    host_call_ms = [0.0] * G

    def drive(g):
        # one host thread per device (the library's own host path does the same: one worker thread per device); every
        # call is an asynchronous enqueue on the device's stream
        s = shards[g]
        torch.cuda.set_device(s["dev"])
        t0 = time.perf_counter()
        for k in range(args.steps):
            evs[g][k][0].record(s["ts"])
            codec.decode_device(fmt, s["packed"], s["p_off"], s["c_len"], s["d_dst"], s["r_off"], s["r_len"], s["olen"], s["cons"], s["st"],
                                device=g, stream=s["ts"].cuda_stream)
            evs[g][k][1].record(s["ts"])
        host_call_ms[g] = (time.perf_counter() - t0) * 1e3 / args.steps

    if G == 1:
        drive(0)
    else:
        import threading
        th = [threading.Thread(target=drive, args=(g,)) for g in range(G)]
        for t in th:
            t.start()
        for t in th:
            t.join()
    sync_all()
    barrier()
    t_wall1 = time.time()
    launches = codec.kernel_launches - launches0
    clocks = sampler.stop(t_wall0, t_wall1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, shards, n, size)
    total_ms = max(ev[0][0].elapsed_time(ev[-1][1]) for ev in evs)              # max over devices
    kernel_ms = sum(a.elapsed_time(b) for a, b in evs[0]) / args.steps            # device 0: the roofline kernel
    ms_per_step = total_ms / args.steps
    value = G * out_bytes / (ms_per_step * 1e-3) / 1e9

    # ---- per-class device timing on device 0 (outside the headline region; explains the mix)
    s0 = shards[0]
    torch.cuda.set_device(s0["dev"])
    dev, ts = s0["dev"], s0["ts"]
    per_class = {}
    cls_idx = {c: torch.tensor([i for i, k in enumerate(s0["classes"]) if k == c], device=dev) for c in sorted(set(s0["classes"]))}
    for c, ix in cls_idx.items():
        po, cl, ro, rl = s0["p_off"][ix].contiguous(), s0["c_len"][ix].contiguous(), s0["r_off"][ix].contiguous(), s0["r_len"][ix].contiguous()
        best, _, _ = time_decode(codec, fmt, s0["packed"], po, cl, s0["d_dst"], ro, rl, opts, 3, 1, ts)
        cb, ob = int(cl.sum()), len(ix) * size
        per_class[c] = {"streams": len(ix), "ratio": round(cb / ob, 4), "out_gbs": round(ob / best / 1e6, 1), "hbm_gbs": round((cb + ob) / best / 1e6, 1)}

    # ---- end to end through the C ABI with pinned host buffers (H2D + kernel + D2H inside the timed region): ONE
    #      aurora_decode_batch call over the streams of all devices; the library cuts the batch into per-device shards
    L = _lib.load()
    src_total = sum(s["comp_total"] for s in shards)
    h_src_p = L.aurora_pinned_alloc(src_total + 16)
    h_dst_p = L.aurora_pinned_alloc(G * out_bytes + 16)
    assert h_src_p and h_dst_p, "pinned allocation failed"
    h_src = np.ctypeslib.as_array(C.cast(h_src_p, C.POINTER(C.c_uint8)), shape=(src_total + 16,))
    h_dst = np.ctypeslib.as_array(C.cast(h_dst_p, C.POINTER(C.c_uint8)), shape=(G * out_bytes + 16,))
    h_off, h_len, base = [], [], 0
    for s in shards:
        torch.from_numpy(h_src[base:base + s["comp_total"]]).copy_(s["packed"][:s["comp_total"]])
        h_off.append(s["p_off"].cpu().numpy().astype(np.uint64) + np.uint64(base))
        h_len.append(s["c_len"].cpu().numpy().astype(np.uint64))
        base += s["comp_total"]
    h_off, h_len = np.concatenate(h_off), np.concatenate(h_len)
    h_doff = np.arange(G * n, dtype=np.uint64) * np.uint64(size)
    h_cap = np.full(G * n, size, dtype=np.uint64)
    e2e_steps = args.steps
    for _ in range(2):
        out_len, consumed, status = codec.decode_packed(fmt, h_src, h_off, h_len, h_dst, h_doff, h_cap, opts)
    assert (status == 0).all()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        out_len, consumed, status = codec.decode_packed(fmt, h_src, h_off, h_len, h_dst, h_doff, h_cap, opts)
    for s in shards:
        torch.cuda.synchronize(s["dev"])
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    barrier()
    e2e_ok = bool((status == 0).all())
    for g, s in enumerate(shards):
        e2e_ok = e2e_ok and bool(np.array_equal(h_dst[g * out_bytes:(g + 1) * out_bytes], s["raw"].view(-1).cpu().numpy()))
    e2e_value = G * out_bytes / e2e_s / 1e9
    h2d = src_total + 4 * 8 * G * n
    d2h = G * out_bytes + G * n * (8 + 8 + 4)

    # ---- CPU baseline (N == 1 only): the oracle on a bounded sample of the same streams
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        O.build()
        threads = O.hardware_threads()
        sample = min(n, 16384)
        cdst = np.zeros(sample * size + 16, dtype=np.uint8)
        best = 1e30
        for _ in range(3):
            t0 = time.perf_counter()
            ol, co, st_ = O.decode_packed(fmt, h_src, h_off[:sample], h_len[:sample], cdst, h_doff[:sample], h_cap[:sample], None, threads)
            best = min(best, time.perf_counter() - t0)
        assert (st_ == 0).all() and np.array_equal(cdst[:sample * size], h_dst[:sample * size]), "oracle and GPU disagree"
        cpu_baseline = {"value": round(sample * size / best / 1e9, 3), "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"first {sample} of the {n} streams ({sample * size >> 20} MiB decoded), best of 3, std::thread over {threads} host threads",
                        "note": "C++ restatement of the reference's managed decoder (no .NET runtime on the box)"}
    L.aurora_pinned_free(h_src_p)
    L.aurora_pinned_free(h_dst_p)
    del h_src, h_dst

    # ---- the other configs of the metric (N == 1): device 0
    configs = None
    if world == 1 and not args.no_configs:
        raw_c2 = s0["raw"]
        for s in shards:
            for k in ("packed", "d_dst"):
                s[k] = None
        torch.cuda.empty_cache()
        configs = other_configs(codec, dev, ts, peak, raw_c2, args)

    achieved = (s0["comp_bytes"] + out_bytes) / (kernel_ms * 1e-3) / 1e9
    traffic, capture = ncu_traffic("lz10_c2", n)
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
        "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "config": workload_config(n, world),
        "roofline": {"bound": "hbm", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                     "traffic": traffic, "traffic_source": capture, "peak_source": peak_src, "kernel": "decode_flaglz_kernel<LZ10>",
                     "algorithmic_bytes_per_launch": s0["comp_bytes"] + out_bytes, "kernel_ms": round(kernel_ms, 4)},
        "cpu_baseline": cpu_baseline,
        "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "verified": e2e_ok, "steps": e2e_steps, "devices_in_context": G,
                "path": "one aurora_decode_batch call; the library shards the batch over its per-device worker threads"},
        "gpu_launches": int(launches),
        "host_enqueue_ms_per_step": [round(v, 3) for v in host_call_ms],
        "clocks": clocks,
        "per_class": per_class,
        "compression_ratio": round(comp_bytes / (G * out_bytes), 4),
        "encode_s": round(t_enc, 3),
        "configs": configs,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    codec.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed passes over the C2 batch, both device resident (value) and end to end (e2e); the per-class "
                         "breakdown and the configs C3 / C4 / C5 time fixed counts of their own")
    ap.add_argument("--warmup", type=int, default=3,
                    help="untimed decode passes before the timed steps (the GPU arm runs at least 3: its line's warmup says how many)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--streams", type=int, default=FULL_STREAMS, help="streams per GPU (default: the full C2 configuration)")
    ap.add_argument("--c3-streams", type=int, default=16384, help="streams of config C3 (all three formats together)")
    ap.add_argument("--c4-streams", type=int, default=1 << 20, help="streams of config C4 (each of the three formats)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="headline only (skip C3 / C4 / C5)")
    ap.add_argument("--quick", action="store_true", help="C5 only among the other configs")
    ap.add_argument("--dump-batch", default=None, help="write the reference arm's C2 sample (packed.bin, index.bin) for baseline/dotnet and exit")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one decoded to DIR/*.npy (float32 / float64, at most 64 MB): "
                         "status, out_len, consumed and a digest of the decoded bytes of every stream, and the bytes of a fixed "
                         "sample of streams")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl == "reference" or args.dump_batch):
        ap.error("--dump-outputs writes the outputs of the GPU decode (--impl ours)")
    if args.impl == "reference" or args.dump_batch:
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
