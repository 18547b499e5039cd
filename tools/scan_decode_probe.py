"""Times the CLI's `-scan` walk over a device image three ways, alternated in one process (DESIGN.md §4.5):
  (a) BatchCodec.scan_decode_device — the walk on the device, in rounds;
  (b) scan_offsets_device, the bitmap to the host, and one decode_device per visited hit (the route without (a));
  (c) one decode_device of the known asset starts: the floor (no IsMatch, no walk).
The image (at least 1 GiB, larger than L2) holds C2-shaped Yaz0, LZ10 and LZ4 assets between random junk; each format's walk finds
its own assets.  (a) and (b) must return the same entries before anything is timed.  Writes one JSON file with the card's name
and power limit.

    python tools/scan_decode_probe.py --out profiles/scan_decode_probe.json [--image-mib 1024] [--assets 2048] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from auroralib.compression_b200 import BatchCodec, _abi as A  # noqa: E402
from auroralib.compression_b200.corpus import generate_mix  # noqa: E402

FORMATS = [(A.FMT_YAZ0, "Yaz0"), (A.FMT_LZ10, "LZ10"), (A.FMT_LZ4, "LZ4")]
RAW = 1 << 16   # C2: 64 KiB streams
MAX_SIZE = 1 << 26


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=60).stdout.strip()
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # the card name still comes from torch
        return torch.cuda.get_device_name(0), f"unknown ({e})"


def build_image(codec, image_bytes, n_assets, seed):
    """-> (device image, {fmt: (starts, raw tensors)})"""
    rng = np.random.default_rng(seed)
    comps = {}
    for fmt, _ in FORMATS:
        raw, _ = generate_mix(n_assets, RAW, seed=seed + fmt)
        blobs = [raw[i].numpy().tobytes() for i in range(n_assets)]
        c, st = codec.encode_batch(fmt, blobs, A.make_opts(quality=8))
        assert (st == 0).all()
        comps[fmt] = (c, raw)
    order = [(fmt, i) for fmt, _ in FORMATS for i in range(n_assets)]
    rng.shuffle(order)
    total_comp = sum(len(comps[f][0][i]) for f, i in order)
    gap = max(64, (image_bytes - total_comp) // len(order))
    g = torch.Generator(device="cuda").manual_seed(seed)
    img = torch.randint(0, 256, (image_bytes + (1 << 20),), dtype=torch.uint8, device="cuda", generator=g)
    starts = {fmt: [] for fmt, _ in FORMATS}
    idx = {fmt: [] for fmt, _ in FORMATS}
    pos = 0
    for fmt, i in order:
        pos += int(rng.integers(gap // 2, gap * 3 // 2))
        pos = (pos + 15) & ~15   # 16-byte aligned starts keep (b) and (c) inside decode_device's offset rule
        c = comps[fmt][0][i]
        img[pos:pos + len(c)] = torch.frombuffer(bytearray(c), dtype=torch.uint8).cuda()
        starts[fmt].append(pos)
        idx[fmt].append(i)
        pos += len(c)
    length = max(pos + 4096, image_bytes)
    img = img[:length].clone()
    return img, {fmt: (starts[fmt], comps[fmt][1][idx[fmt]]) for fmt, _ in FORMATS}


def walk_a(codec, fmt, img):
    return codec.scan_decode_device(fmt, img, max_size=MAX_SIZE)


def walk_b(codec, fmt, img):
    """scan_offsets_device, the bitmap to the host, one decode_device per visited hit (its window [h, len), capacity max_size)."""
    n = img.numel()
    match = torch.empty(n, dtype=torch.uint8, device="cuda")
    st_ = torch.cuda.current_stream().cuda_stream   # the library calls run on torch's stream, ordered with its tensors
    codec.scan_offsets_device(fmt, img, match, stream=st_)
    hits = np.nonzero(match.cpu().numpy())[0]
    one = torch.zeros(1, dtype=torch.int64, device="cuda")
    cap = torch.full((1,), MAX_SIZE, dtype=torch.int64, device="cuda")
    dst = torch.empty(MAX_SIZE, dtype=torch.uint8, device="cuda")
    out_len = torch.empty(1, dtype=torch.int64, device="cuda")
    consumed = torch.empty(1, dtype=torch.int64, device="cuda")
    status = torch.empty(1, dtype=torch.int32, device="cuda")
    entries, outs, i, k = [], [], 0, 0
    while True:
        k = int(np.searchsorted(hits, i, side="left"))
        if k >= len(hits):
            break
        h = int(hits[k])
        off = torch.full((1,), h, dtype=torch.int64, device="cuda")
        ln = torch.full((1,), n - h, dtype=torch.int64, device="cuda")
        codec.decode_device(fmt, img, off, ln, dst, one, cap, out_len, consumed, status, stream=st_)
        st, c, ol = int(status[0]), int(consumed[0]), int(out_len[0])
        if st == A.OK:
            entries.append((h, c, ol))
            outs.append(dst[:ol].clone())
            i = h + max(c, 1)
        else:
            i = h + 1
    return entries, outs


def decode_c(codec, fmt, img, starts):
    n = len(starts)
    off = torch.tensor(starts, dtype=torch.int64, device="cuda")
    ln = img.numel() - off
    cap = torch.full((n,), RAW, dtype=torch.int64, device="cuda")
    doff = torch.arange(n, dtype=torch.int64, device="cuda") * RAW
    dst = torch.empty(n * RAW, dtype=torch.uint8, device="cuda")
    out_len = torch.empty(n, dtype=torch.int64, device="cuda")
    consumed = torch.empty(n, dtype=torch.int64, device="cuda")
    status = torch.empty(n, dtype=torch.int32, device="cuda")
    codec.decode_device(fmt, img, off, ln, dst, doff, cap, out_len, consumed, status, stream=torch.cuda.current_stream().cuda_stream)
    return status, dst


def timed(f):
    torch.cuda.synchronize()
    t = time.perf_counter()
    r = f()
    torch.cuda.synchronize()
    return time.perf_counter() - t, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--image-mib", type=int, default=1024)
    ap.add_argument("--assets", type=int, default=2048, help="assets per format")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("scan_decode_probe: no CUDA device (this probe measures the GPU only)")
    # a stream of its own: handle 0 (torch's legacy default stream) would mean the library's own stream to the C ABI, which is
    # not ordered with torch's work
    torch.cuda.set_stream(torch.cuda.Stream())
    codec = BatchCodec()
    name, power = card()
    img, truth = build_image(codec, args.image_mib << 20, args.assets, 0x5CA7)
    result = {"card": name, "power_limit": power, "image_bytes": img.numel(), "assets_per_format": args.assets, "raw_asset_bytes": RAW,
              "max_size": MAX_SIZE, "reps": args.reps, "formats": {}}
    for fmt, fname in FORMATS:
        starts, raw = truth[fmt]
        # correctness first: (a) and (b) give the same entries, and every asset is among them
        st, c, ol, dst, off = walk_a(codec, fmt, img)
        ea = list(zip(st.tolist(), c.tolist(), ol.tolist()))
        eb, outs = walk_b(codec, fmt, img)
        assert ea == eb, (fname, len(ea), len(eb))
        for k, o in enumerate(off.tolist()):
            assert torch.equal(dst[o:o + ea[k][2]], outs[k]), (fname, k)
        assert set(starts) <= set(st.tolist()), fname
        sc, dc = decode_c(codec, fmt, img, starts)
        assert (sc == 0).all() and torch.equal(dc.view(len(starts), RAW), raw.cuda()), fname
        codec.scan_offsets_device(fmt, img, torch.empty(img.numel(), dtype=torch.uint8, device="cuda"), stream=torch.cuda.current_stream().cuda_stream)
        times = {"a": [], "b": [], "c": [], "scan_offsets": []}
        match = torch.empty(img.numel(), dtype=torch.uint8, device="cuda")
        for _ in range(args.reps):
            times["a"].append(timed(lambda: walk_a(codec, fmt, img))[0])
            times["b"].append(timed(lambda: walk_b(codec, fmt, img))[0])
            times["c"].append(timed(lambda: decode_c(codec, fmt, img, starts))[0])
            times["scan_offsets"].append(timed(lambda: codec.scan_offsets_device(fmt, img, match, stream=torch.cuda.current_stream().cuda_stream))[0])
        med = {k: float(np.median(v)) for k, v in times.items()}
        result["formats"][fname] = {"entries": len(ea), "seconds_median": med, "seconds_all": times,
                                    "a_over_c_plus_scan": med["a"] / (med["c"] + med["scan_offsets"]), "b_over_a": med["b"] / med["a"]}
        print(fname, json.dumps(result["formats"][fname]["seconds_median"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"card": name, "power_limit": power, "formats": {k: v["seconds_median"] for k, v in result["formats"].items()}}))


if __name__ == "__main__":
    main()
