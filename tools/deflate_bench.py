"""Device deflate of the coefficient streams (aeaj_deflate_coefficients) on one GPU, in one run:
  (a) kernel time (CUDA events) of deflate on the bench's 16-frame 4K C2 sub-batch (encode(stream=True) first): input GB/s,
      output bytes against zlib level 9 on the same streams;
  (b) Jpeg.compress_batch on bench.py's compress_full workload (8 x 1080p, YCoCg q40-80 b4-64), deflate="host" against
      deflate="device", alternated and repeated: MP/s and total bytes.
Prints one JSON object (and writes it to --out if given).  Usage: python tools/deflate_bench.py [--out FILE] [--reps N]"""
import argparse
import json
import os
import subprocess
import sys
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "adaptive-edge-aware-jpeg_b200"), os.path.join(ROOT, "tests"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

import bench


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def kernel_leg(codec, reps):
    B = 16
    rgb = torch.from_numpy(bench.frames_u8(range(B), bench.H, bench.W, os.cpu_count() or 1)).cuda()
    s, q, b = bench.SPACE, bench.QRANGE, bench.BRANGE
    enc = codec.encode(rgb, s, q, b, stream=True)
    df = codec.deflate(enc, s, q, b)                               # warm-up: buffers, descriptor table
    torch.cuda.synchronize()
    counts = enc.counts.cpu().numpy()
    nbytes = int(counts[:, :, 2].sum()) * 4
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        e0.record()
        codec.deflate(enc, s, q, b)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    lengths = df.lengths.cpu().numpy()
    dev_bytes = int(lengths.sum())
    raws = [enc.coef[l][i, :int(counts[i, l, 2])].cpu().numpy().tobytes() for i in range(B) for l in range(3)]
    with ThreadPoolExecutor(os.cpu_count() or 1) as pool:
        z9 = sum(pool.map(lambda r: len(zlib.compress(r, 9)), raws))
    ok = all(zlib.decompress(df.out[l][i, :int(lengths[i, l])].cpu().numpy().tobytes()) == raws[i * 3 + l]
             for i in range(B) for l in range(3))
    ms = float(np.median(times))
    return {"workload": f"{B} x {bench.W}x{bench.H} C2 ({s} q{q[0]}-{q[1]} b{b[0]}-{b[1]}), encode(stream=True) then deflate",
            "input_bytes": nbytes, "deflate_ms_median": ms, "deflate_ms_all": times, "input_gb_s": nbytes / ms / 1e6,
            "device_bytes": dev_bytes, "zlib9_bytes": z9, "ratio_vs_zlib9": dev_bytes / z9, "round_trip_ok": ok}


def compress_leg(reps):
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    imgs = [Image.from_uint8(fr, ".png") for fr in bench.frames_u8(range(8), 1080, 1920, os.cpu_count() or 1)]
    st = JpegCompressionSettings("YCoCg", (40, 80), (4, 64))
    coders = {"host": Jpeg(st), "device": Jpeg(st, deflate="device")}
    for j in coders.values():
        j.compress_batch(imgs[:2])
        j.compress_batch(imgs)
    mp = len(imgs) * 1080 * 1920 / 1e6
    res = {k: {"mp_s": [], "bytes": None} for k in coders}
    blobs = {}
    for _ in range(reps):
        for k, j in coders.items():
            t0 = time.perf_counter()
            blobs[k] = j.compress_batch(imgs)
            res[k]["mp_s"].append(mp / (time.perf_counter() - t0))
            res[k]["bytes"] = int(sum(map(len, blobs[k])))
    dec = [Jpeg(st).decompress_batch(blobs[k], as_uint8=True) for k in coders]
    for k in coders:
        res[k]["mp_s_median"] = float(np.median(res[k]["mp_s"]))
    return {"workload": "8 synthetic 1920x1080 frames, YCoCg q40-80 b4-64, Jpeg.compress_batch incl. .ajpg framing, wall clock, "
                        "host / device alternated", "host_threads": os.cpu_count(), **res,
            "speedup": res["device"]["mp_s_median"] / res["host"]["mp_s_median"],
            "bytes_ratio": res["device"]["bytes"] / res["host"]["bytes"],
            "decoded_equal": all(np.array_equal(a, b_) for a, b_ in zip(dec[0], dec[1]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the result to this file")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("deflate_bench needs a CUDA device")
    from aeaj.codec import get_codec
    codec = get_codec(0)
    res = {"gpu": card(), "kernel": kernel_leg(codec, 3 * args.reps), "compress_full": compress_leg(args.reps)}
    print(json.dumps(res), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
