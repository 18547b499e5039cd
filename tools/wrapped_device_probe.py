"""What decoding wrapped streams on the device costs (aurora_decode_batch_device for the wrapper formats).

On one GPU, C2-shaped files (64 KiB each of the C2 mix, corpus.generate_mix) are encoded by the engine five ways and decoded
with BatchCodec.decode_device, timed with CUDA events on the launching stream:
  (a) bare LZ10;
  (b) GCLZ: the same LZ10 streams behind a 4-byte header, so every sub-stream starts 4 bytes past a 16-byte boundary;
  (c) Level5: headerless LZ10 bodies behind the 4-byte Level5 word;
  (d) LZ77 ChunkLZ10 with 4 KiB chunks: 16 times as many (smaller) sub-streams, plus the call's one host read of the chunk
      count.  Files whose chunk ends do not fit u16 are refused by the encoder; only the files it accepts are kept;
  (e) LZ00 (Lzss0 body under the keystream, lifted into per-stream scratch slots after one host read of their total) against
      bare LZSS with the same properties.
Every result is checked against the raw bytes.  The card's name, power limit and SM clock are read in the same process.
Writes one JSON line to stdout and, with --out, to a file.

    python tools/wrapped_device_probe.py --out profiles/wrapped_device_probe.json
    python tools/wrapped_device_probe.py --only e_lzss_lzss0,e_lz00     (some shapes only)
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.device_query_probe import card, event_ms  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--files", type=int, default=16384)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default=None, help="comma-separated shape names (default: all)")
    args = ap.parse_args()

    import numpy as np
    import torch
    from auroralib.compression_b200 import BatchCodec, corpus, layout, pack
    from auroralib.compression_b200 import _abi as A
    if not torch.cuda.is_available():
        raise SystemExit("wrapped_device_probe: no CUDA device (these numbers exist only on the GPU)")
    dev = torch.device("cuda", 0)
    codec = BatchCodec(device_mask=1)
    ts = torch.cuda.Stream(device=dev)
    res = {"card": card(), "iters": args.iters, "file_bytes": 65536}

    n, size = args.files, 65536
    raw, _ = corpus.generate_mix(n, size, device=dev)
    raw = raw.reshape(n, size)
    raw_h = raw.cpu().numpy()
    raws = [raw_h[i].tobytes() for i in range(n)]
    lzss0 = A.lz_props_window(0x1000, 0xF + 3, 3, 0xFEE)
    shapes = [
        ("a_lz10", A.FMT_LZ10, A.make_opts(quality=8)),
        ("b_gclz", A.FMT_GCLZ, A.make_opts(quality=8)),
        ("c_level5", A.FMT_LEVEL5, A.make_opts(quality=8)),
        ("d_lz77_chunklz10_4k", A.FMT_LZ77, A.make_opts(quality=8, lz77_type=0xF7, lz77_chunk_size=0x1000)),
        ("e_lzss_lzss0", A.FMT_LZSS, A.make_opts(quality=8, lzss=lzss0)),
        ("e_lz00", A.FMT_LZ00, A.make_opts(quality=8, lz00_key=0x5EEDC0DE)),
    ]
    if args.only:
        shapes = [x for x in shapes if x[0] in args.only.split(",")]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a).astype(np.int64)).to(dev)
    for name, fmt, opts in shapes:
        comps, st = codec.encode_batch(fmt, raws, opts)
        keep = [i for i in range(n) if st[i] == 0]
        base, off, ln = pack([comps[i] for i in keep])
        caps, doff, total = layout([size] * len(keep))
        m = len(keep)
        d_src, d_off, d_len = torch.from_numpy(base).to(dev), t(off), t(ln)
        d_doff, d_cap = t(doff), t(caps)
        d_dst = torch.empty(total + 16, dtype=torch.uint8, device=dev)
        d_olen = torch.empty(m, dtype=torch.int64, device=dev)
        d_cons = torch.empty(m, dtype=torch.int64, device=dev)
        d_st = torch.empty(m, dtype=torch.int32, device=dev)
        torch.cuda.synchronize(dev)
        # the decode of the same options as the encode (LZSS: the Lzss0 properties; the wrappers fix their own)
        call = lambda: codec.decode_device(fmt, d_src, d_off, d_len, d_dst, d_doff, d_cap, d_olen, d_cons, d_st, opts, stream=ts.cuda_stream)
        before = codec.kernel_launches
        with torch.cuda.stream(ts):
            call()
            ts.synchronize()
            launches = codec.kernel_launches - before
            ms = event_ms(call, ts, args.iters, 3)
        want = raw[torch.tensor(keep, device=dev)]
        ok = int((d_st == 0).sum()) == m and torch.equal(d_olen, d_cap) and torch.equal(d_dst[:m * size].view(m, size), want)
        assert ok, name
        res[name] = {"format_id": fmt, "files": m,
                     "files_refused_by_encoder": n - m, "raw_bytes": m * size, "comp_bytes": int(ln.sum()),
                     "launches_per_call": launches, "ms_per_step": round(ms, 4),
                     "decoded_gbps": round(m * size / (ms * 1e-3) / 1e9, 1)}
        del d_src, d_dst, comps
        torch.cuda.empty_cache()
    for k in ("b_gclz", "c_level5", "d_lz77_chunklz10_4k"):
        if k in res and "a_lz10" in res:
            res[k]["rate_vs_a"] = round(res[k]["decoded_gbps"] / res["a_lz10"]["decoded_gbps"], 3)
    if "e_lz00" in res and "e_lzss_lzss0" in res:
        res["e_lz00"]["rate_vs_bare_lzss"] = round(res["e_lz00"]["decoded_gbps"] / res["e_lzss_lzss0"]["decoded_gbps"], 3)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
