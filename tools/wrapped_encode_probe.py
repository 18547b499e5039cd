"""What encoding wrapped streams on the device costs (aurora_encode_batch_device for the wrapper formats).

On one GPU, C2-shaped files (64 KiB each of the C2 mix, corpus.generate_mix) are encoded at quality 8 with
BatchCodec.encode_device, timed with CUDA events on the launching stream over warmed calls:
  (1) bare LZ10;
  (2) GCLZ: the same LZ10 streams behind a 4-byte header (plan pass, LZ10, finish pass);
  (3) Level5: LZ10 with its header rewritten in place;
  (4) LZ77 ChunkLZ10 with 4 KiB chunks: 16 times as many core streams, the compaction, plus the call's one host read of the
      chunk count;
  (5) LZ00 (Lzss0 body under the keystream) against bare LZSS with the same properties;
  (6) the route a device-resident caller had for GCLZ before: the raw tensor copied to the host, aurora_encode_batch, the
      packed outputs copied back to the device (wall clock, every step waited for).
Every output is checked against the host entry point (status, out_len, bytes) before it is timed.  The card's name, power
limit and SM clock are read in the same process.  Writes one JSON line to stdout and, with --out, to a file.

    python tools/wrapped_encode_probe.py --out profiles/wrapped_encode_probe.json
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.device_query_probe import card, event_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--files", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--host-iters", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch
    from auroralib.compression_b200 import BatchCodec, corpus, layout
    from auroralib.compression_b200 import _abi as A
    if not torch.cuda.is_available():
        raise SystemExit("wrapped_encode_probe: no CUDA device (these numbers exist only on the GPU)")
    dev = torch.device("cuda", 0)
    codec = BatchCodec(device_mask=1)
    ts = torch.cuda.Stream(device=dev)
    res = {"card": card(), "iters": args.iters, "file_bytes": 65536, "quality": 8}

    n, size = args.files, 65536
    raw, _ = corpus.generate_mix(n, size, device=dev)
    raw = raw.reshape(-1).contiguous()
    raw_h = raw.cpu().numpy()
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a).astype(np.int64)).to(dev)
    off = np.arange(n, dtype=np.uint64) * size
    ln = np.full(n, size, dtype=np.uint64)
    d_off, d_len = t(off), t(ln)
    lzss0 = A.lz_props_window(0x1000, 0xF + 3, 3, 0xFEE)
    shapes = [
        ("1_lz10", A.FMT_LZ10, A.make_opts(quality=8)),
        ("2_gclz", A.FMT_GCLZ, A.make_opts(quality=8)),
        ("3_level5", A.FMT_LEVEL5, A.make_opts(quality=8)),
        ("4_lz77_chunklz10_4k", A.FMT_LZ77, A.make_opts(quality=8, lz77_type=0xF7, lz77_chunk_size=0x1000)),
        ("5_lzss_lzss0", A.FMT_LZSS, A.make_opts(quality=8, lzss=lzss0)),
        ("5_lz00", A.FMT_LZ00, A.make_opts(quality=8, lz00_key=0x5EEDC0DE)),
    ]
    for name, fmt, opts in shapes:
        caps, doff, total = layout([codec.encode_bound(fmt, size)] * n)
        d_doff, d_cap = t(doff), t(caps)
        d_dst = torch.empty(total + 16, dtype=torch.uint8, device=dev)
        d_olen = torch.empty(n, dtype=torch.int64, device=dev)
        d_st = torch.empty(n, dtype=torch.int32, device=dev)
        torch.cuda.synchronize(dev)
        call = lambda: codec.encode_device(fmt, raw, d_off, d_len, d_dst, d_doff, d_cap, d_olen, d_st, opts, stream=ts.cuda_stream)
        before = codec.kernel_launches
        with torch.cuda.stream(ts):
            call()
            ts.synchronize()
        launches = codec.kernel_launches - before
        # the host entry point on the same inputs: statuses, lengths and bytes must agree
        h_dst = np.zeros(total + 16, dtype=np.uint8)
        h_olen, h_st = codec.encode_packed(fmt, raw_h, off, ln, h_dst, doff, caps, opts)
        g_dst, g_olen, g_st = d_dst.cpu().numpy(), d_olen.cpu().numpy(), d_st.cpu().numpy()
        assert (g_st == h_st).all() and (g_olen.astype(np.uint64) == h_olen).all(), name
        for i in np.nonzero(h_st == 0)[0]:
            a, b = int(doff[i]), int(doff[i]) + int(h_olen[i])
            assert np.array_equal(g_dst[a:b], h_dst[a:b]), (name, int(i))
        with torch.cuda.stream(ts):
            ms = event_ms(call, ts, args.iters, 3)
        ok = int((h_st == 0).sum())
        res[name] = {"format_id": fmt, "files": n, "files_ok": ok, "raw_bytes": n * size,
                     "comp_bytes_ok": int(h_olen[h_st == 0].sum()), "launches_per_call": launches, "ms_per_call": round(ms, 4),
                     "raw_gbps_in": round(n * size / (ms * 1e-3) / 1e9, 2)}
        if name == "2_gclz":
            # (6) the host route: raw to the host, aurora_encode_batch, the packed outputs back to the device
            pinned = torch.empty(n * size, dtype=torch.uint8).pin_memory()
            out_h = np.zeros(total + 16, dtype=np.uint8)

            def host_route():
                pinned.copy_(raw, non_blocking=True)
                torch.cuda.synchronize(dev)
                olen, st = codec.encode_packed(fmt, pinned.numpy(), off, ln, out_h, doff, caps, opts)
                back = torch.from_numpy(out_h).to(dev, non_blocking=False)
                torch.cuda.synchronize(dev)
                return back, olen, st

            host_route()
            times = []
            for _ in range(args.host_iters):
                t0 = time.perf_counter()
                host_route()
                times.append((time.perf_counter() - t0) * 1e3)
            hms = float(np.median(times))
            res["6_gclz_host_route"] = {"format_id": fmt, "files": n, "ms_per_call": round(hms, 3),
                                        "raw_gbps_in": round(n * size / (hms * 1e-3) / 1e9, 2),
                                        "timing": f"wall clock, median of {args.host_iters}"}
        del d_dst
        torch.cuda.empty_cache()
    a = res["1_lz10"]["raw_gbps_in"]
    for k in ("2_gclz", "3_level5", "4_lz77_chunklz10_4k"):
        res[k]["rate_vs_1"] = round(res[k]["raw_gbps_in"] / a, 3)
    res["5_lz00"]["rate_vs_bare_lzss"] = round(res["5_lz00"]["raw_gbps_in"] / res["5_lzss_lzss0"]["raw_gbps_in"], 3)
    res["6_gclz_host_route"]["time_vs_2"] = round(res["6_gclz_host_route"]["ms_per_call"] / res["2_gclz"]["ms_per_call"], 2)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
