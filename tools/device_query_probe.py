"""What finding the decoded sizes on the device costs (aurora_decoded_size_batch_device and BatchCodec.decode_device_sized).

On one GPU, with CUDA events on the launching stream:
  * the header peek of decoded_size_device on the C2 batch (65 536 LZ10 streams x 64 KiB of the C2 mix);
  * an LZ4 block size scan on a C4-shaped batch (ragged 4 - 64 KiB streams of classes T / M / X), next to a decode of the same
    batch with known capacities (the size scan is the decode parser with its stores dropped);
  * decode_device_sized (peek + capacity prefix sum + one host read of the total + allocation + decode) against decode_device
    with known capacities on C2, wall clock from the launch to a stream synchronise; the difference is the cost of not
    knowing the sizes.
Every result is checked (statuses, sizes, decoded bytes).  The card's name, power limit and SM clock are read in the same
process.  Writes one JSON line to stdout and, with --out, to a file.

    python tools/device_query_probe.py --out profiles/device_query_probe.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        line = subprocess.check_output(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], text=True).strip()
    except (OSError, subprocess.CalledProcessError) as e:
        return {"error": str(e)}
    return dict(zip(q.split(","), [v.strip() for v in line.split(",")]))


def event_ms(fn, ts, iters, warmup):
    """Average ms of fn() over `iters` back-to-back launches on `ts` (after `warmup` calls)."""
    import torch
    for _ in range(warmup):
        fn()
    ts.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(ts)
    for _ in range(iters):
        fn()
    b.record(ts)
    ts.synchronize()
    return a.elapsed_time(b) / iters


def wall_ms(fn, ts, iters, warmup):
    """Median wall-clock ms of fn() followed by a synchronise of `ts`."""
    for _ in range(warmup):
        fn()
        ts.synchronize()
    t = []
    for _ in range(iters):
        t0 = time.perf_counter()
        fn()
        ts.synchronize()
        t.append((time.perf_counter() - t0) * 1e3)
    t.sort()
    return t[len(t) // 2]


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--c2-streams", type=int, default=65536)
    ap.add_argument("--c4-streams", type=int, default=1 << 18)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import bench
    from auroralib.compression_b200 import BatchCodec, corpus
    from auroralib.compression_b200 import _abi as A
    if not torch.cuda.is_available():
        raise SystemExit("device_query_probe: no CUDA device (these numbers exist only on the GPU)")
    dev = torch.device("cuda", 0)
    codec = BatchCodec(device_mask=1)
    ts = torch.cuda.Stream(device=dev)
    res = {"card": card(), "iters": args.iters}

    # ---- C2: 65 536 LZ10 streams x 64 KiB
    n, size = args.c2_streams, 65536
    raw, _ = corpus.generate_mix(n, size, device=dev)
    raw = raw.reshape(-1)
    r_off = torch.arange(n, dtype=torch.int64, device=dev) * size
    r_len = torch.full((n,), size, dtype=torch.int64, device=dev)
    packed, p_off, c_len, comp_total, _ = bench.gpu_encode(codec, A.FMT_LZ10, raw, r_off, r_len, A.make_opts(quality=8), dev, ts)
    d_size = torch.empty(n, dtype=torch.int64, device=dev)
    d_sst = torch.empty(n, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    with torch.cuda.stream(ts):
        peek = event_ms(lambda: codec.decoded_size_device(A.FMT_LZ10, packed, p_off, c_len, d_size, d_sst, stream=ts.cuda_stream),
                        ts, 10 * args.iters, 5)
    assert int((d_sst != 0).sum()) == 0 and torch.equal(d_size, r_len)
    res["c2_header_peek"] = {"streams": n, "ms": round(peek, 4), "launches_per_call": 1}

    d_dst = torch.empty(n * size + 16, dtype=torch.uint8, device=dev)
    d_olen = torch.empty(n, dtype=torch.int64, device=dev)
    d_cons = torch.empty(n, dtype=torch.int64, device=dev)
    d_st = torch.empty(n, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)

    def known():
        codec.decode_device(A.FMT_LZ10, packed, p_off, c_len, d_dst, r_off, r_len, d_olen, d_cons, d_st, stream=ts.cuda_stream)

    sized_out = []

    def sized():
        sized_out[:] = [codec.decode_device_sized(A.FMT_LZ10, packed, p_off, c_len, stream=ts.cuda_stream)]

    with torch.cuda.stream(ts):
        known_ev = event_ms(known, ts, args.iters, 3)
        # alternate the two so that clock drift and neighbours hit both alike
        kw, sw = [], []
        for _ in range(3):
            kw.append(wall_ms(known, ts, args.iters, 2))
            sw.append(wall_ms(sized, ts, args.iters, 2))
    assert int(d_st.abs().sum()) == 0 and torch.equal(d_dst[:n * size], raw)
    s_dst, s_doff, s_cap, s_olen, s_cons, s_st = sized_out[0]
    assert int(s_st.abs().sum()) == 0 and torch.equal(s_doff, r_off) and torch.equal(s_dst[:n * size], raw)
    del sized_out[:], s_dst
    res["c2_decode"] = {
        "streams": n, "raw_bytes": n * size, "comp_bytes": int(comp_total),
        "decode_device_event_ms": round(known_ev, 3),
        "decode_device_wall_ms": [round(x, 3) for x in kw],
        "decode_device_sized_wall_ms": [round(x, 3) for x in sw],
        "cost_of_unknown_sizes_ms": round(min(sw) - min(kw), 3),
    }
    del packed, d_dst, raw
    torch.cuda.empty_cache()

    # ---- C4-shaped LZ4 block batch: size scan vs decode with known capacities
    m = args.c4_streams
    raw4, o4, l4 = bench.ragged_corpus(m, 4 << 10, 64 << 10, "TMX", 0xA0140000, dev, group=4096)
    packed4, p4, c4, comp4, _ = bench.gpu_encode(codec, A.FMT_LZ4_BLOCK, raw4.view(-1), o4, l4, A.make_opts(quality=8), dev, ts)
    s4 = torch.empty(m, dtype=torch.int64, device=dev)
    st4 = torch.empty(m, dtype=torch.int32, device=dev)
    dst4 = torch.empty(raw4.numel() + 16, dtype=torch.uint8, device=dev)
    ol4 = torch.empty(m, dtype=torch.int64, device=dev)
    co4 = torch.empty(m, dtype=torch.int64, device=dev)
    dst4_st = torch.empty(m, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    with torch.cuda.stream(ts):
        scan_ms = event_ms(lambda: codec.decoded_size_device(A.FMT_LZ4_BLOCK, packed4, p4, c4, s4, st4, size_scan=True,
                                                             stream=ts.cuda_stream), ts, args.iters, 3)
        dec_ms = event_ms(lambda: codec.decode_device(A.FMT_LZ4_BLOCK, packed4, p4, c4, dst4, o4, l4, ol4, co4, dst4_st,
                                                      stream=ts.cuda_stream), ts, args.iters, 3)
    assert int(st4.abs().sum()) == 0 and torch.equal(s4, l4)
    assert int(dst4_st.abs().sum()) == 0 and torch.equal(ol4, l4)
    raw4_bytes = int(l4.sum())
    res["c4_lz4_block"] = {"streams": m, "raw_bytes": raw4_bytes, "comp_bytes": int(comp4),
                           "size_scan_ms": round(scan_ms, 3), "decode_known_caps_ms": round(dec_ms, 3),
                           "size_scan_over_decode": round(scan_ms / dec_ms, 3),
                           "size_scan_gbps_comp_in": round(int(comp4) / (scan_ms * 1e-3) / 1e9, 2),
                           "launches_per_scan": 2}
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
