"""Scaled decode (Jpeg.decompress(..., scale=k), aeaj_decode_scaled) on the B200:
  (a) kernel time (CUDA events, warm-up, median of --reps >= 15) of the device decode at k = 1, 2, 4, 8 from the device-resident
      coefficients of bench.py's 16-frame 4K C2 sub-batch (YCbCr q30-95 b4-128, encode(stream=True) first), uint8 output,
      with the bytes of the uint8 image each call leaves for the download;
  (b) Jpeg.decompress_batch(..., scale=k) on bench.py's compress_full workload (8 x 1080p, YCoCg q40-80 b4-64), wall clock,
      host and device inflate, on files written by each coder.
GPU name and power limit are read in the same run.  Prints one JSON line; --out writes it to profiles/r3_scaled_decode_bench.json
(or the path given).
Usage: python tools/scaled_decode_bench.py [--reps N] [--out [FILE]]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "adaptive-edge-aware-jpeg_b200"), os.path.join(ROOT, "tests"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

import bench

SCALES = (1, 2, 4, 8)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def kernel_leg(codec, reps):
    B = 16
    rgb = torch.from_numpy(bench.frames_u8(range(B), bench.H, bench.W, os.cpu_count() or 1)).cuda()
    s, q, b = bench.SPACE, bench.QRANGE, bench.BRANGE
    enc = codec.encode(rgb, s, q, b, stream=True)
    codec.download(enc)                                             # synchronises, checks the encode
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {"workload": f"{B} x {bench.W}x{bench.H} C2 ({s} q{q[0]}-{q[1]} b{b[0]}-{b[1]}), device-resident coefficients, uint8 out"}
    for k in SCALES:
        def run():
            return codec.decode(enc.coef, enc.leaves, enc.counts, B, bench.H, bench.W, s, q, b, zigzag=True, out="u8", scale=k)
        out = run()                                                 # warm-up: buffers, descriptor tables
        torch.cuda.synchronize()
        codec.check_status(codec.last_decode_status, "decode")
        times = []
        for _ in range(reps):
            e0.record()
            run()
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        res[f"k{k}"] = {"decode_ms_median": float(np.median(times)), "decode_ms_all": times, "launches": codec.last_launches,
                        "out_shape": list(out.shape), "u8_bytes": int(out.numel())}
    return res


def decompress_leg(reps):
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    imgs = [Image.from_uint8(fr, ".png") for fr in bench.frames_u8(range(8), 1080, 1920, os.cpu_count() or 1)]
    st = JpegCompressionSettings("YCoCg", (40, 80), (4, 64))
    files = {"zlib9_files": Jpeg(st).compress_batch(imgs), "device_coded_files": Jpeg(st, deflate="device").compress_batch(imgs)}
    readers = {"host": Jpeg(st), "device": Jpeg(st, deflate="device")}
    mp = len(imgs) * 1080 * 1920 / 1e6
    res = {"workload": "8 synthetic 1920x1080 frames, YCoCg q40-80 b4-64, Jpeg.decompress_batch(scale=k) incl. .ajpg parsing, "
                       "wall clock, megapixels of the full-size frames per second, readers alternated", "host_threads": os.cpu_count()}
    for fk, blobs in files.items():
        r = {}
        for k in SCALES:
            for j in readers.values():
                j.decompress_batch(blobs[:2], scale=k)
                j.decompress_batch(blobs, scale=k)
            t = {name: [] for name in readers}
            for _ in range(reps):
                for name, j in readers.items():
                    t0 = time.perf_counter()
                    j.decompress_batch(blobs, scale=k)
                    t[name].append(mp / (time.perf_counter() - t0))
            r[f"k{k}"] = {f"{name}_mp_s_median": float(np.median(v)) for name, v in t.items()}
        res[fk] = r
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--out", nargs="?", const=os.path.join(ROOT, "profiles", "r3_scaled_decode_bench.json"), default=None,
                    help="also write the result (default path: profiles/r3_scaled_decode_bench.json)")
    args = ap.parse_args()
    if args.reps < 15:
        raise SystemExit("--reps must be at least 15")
    if not torch.cuda.is_available():
        raise SystemExit("scaled_decode_bench needs a CUDA device")
    from aeaj.codec import get_codec
    codec = get_codec(0)
    res = {"gpu": card(), "kernel": kernel_leg(codec, args.reps), "decompress_full": decompress_leg(max(3, args.reps // 3))}
    print(json.dumps(res), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
