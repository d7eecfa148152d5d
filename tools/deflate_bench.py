"""Device deflate / inflate of the coefficient streams (aeaj_deflate_coefficients, aeaj_inflate_coefficients) on one GPU,
in one run:
  deflate legs:
  (a) kernel time (CUDA events) of deflate on the bench's 16-frame 4K C2 sub-batch (encode(stream=True) first): input GB/s,
      output bytes against zlib level 9 on the same streams;
  (b) Jpeg.compress_batch on bench.py's compress_full workload (8 x 1080p, YCoCg q40-80 b4-64), deflate="host" against
      deflate="device", alternated and repeated: MP/s and total bytes.
  inflate legs:
  (c) kernel time (CUDA events) of inflate on the same 4K sub-batch's streams, device-coded and zlib-9 (single segment):
      output GB/s, segments per plane;
  (d) Jpeg.decompress_batch on the compress_full workload, host against device, on files written by each coder (four
      combinations, alternated, medians), and where the host path's time goes: zlib, the int32 upload, the device.
Prints one JSON object (and writes it to --out if given).
Usage: python tools/deflate_bench.py [--out FILE] [--reps N] [--legs deflate,inflate]"""
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


def _plane_args(streams, B):
    """[(b, l, zlib bytes)] -> device zbuf, offsets, lengths"""
    offs, lens = np.zeros((B, 3), np.int64), np.zeros((B, 3), np.int64)
    blob = bytearray()
    for b, l, z in streams:
        offs[b, l], lens[b, l] = len(blob), len(z)
        blob += z
    return [torch.from_numpy(a).cuda() for a in (np.frombuffer(bytes(blob), np.uint8).copy(), offs, lens)]


def inflate_kernel_leg(codec, reps):
    B = 16
    rgb = torch.from_numpy(bench.frames_u8(range(B), bench.H, bench.W, os.cpu_count() or 1)).cuda()
    s, q, b = bench.SPACE, bench.QRANGE, bench.BRANGE
    enc = codec.encode(rgb, s, q, b, stream=True)
    df = codec.deflate(enc, s, q, b)
    torch.cuda.synchronize()
    counts = enc.counts.clone()
    cn = counts.cpu().numpy()
    lengths = df.lengths.cpu().numpy()
    raws = [[enc.coef[l][i, :int(cn[i, l, 2])].cpu().numpy().tobytes() for l in range(3)] for i in range(B)]
    dev_z = [(i, l, df.out[l][i, :int(lengths[i, l])].cpu().numpy().tobytes()) for i in range(B) for l in range(3)]
    with ThreadPoolExecutor(os.cpu_count() or 1) as pool:
        z9 = list(pool.map(lambda il: (il[0], il[1], zlib.compress(raws[il[0]][il[1]], 9)), [(i, l) for i in range(B) for l in range(3)]))
    out_bytes = int(cn[:, :, 2].sum()) * 4
    res = {"workload": f"{B} x {bench.W}x{bench.H} C2 ({s} q{q[0]}-{q[1]} b{b[0]}-{b[1]}) coefficient streams", "output_bytes": out_bytes}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for name, streams in (("device_coded", dev_z), ("zlib9", z9)):
        zbuf, offs, lens = _plane_args(streams, B)
        ib = codec.inflate(zbuf, offs, lens, counts, B, bench.H, bench.W, s, q, b)          # warm-up: buffers, descriptors
        torch.cuda.synchronize()
        times = []
        for _ in range(reps):
            e0.record()
            codec.inflate(zbuf, offs, lens, counts, B, bench.H, bench.W, s, q, b)
            e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        st, seg = ib.status.cpu().numpy(), ib.segments.cpu().numpy()
        ok = bool((st == 0).all()) and all(ib.coef[l][i].view(torch.uint8)[:len(raws[i][l])].cpu().numpy().tobytes() == raws[i][l]
                                           for i in range(B) for l in range(3))
        ms = float(np.median(times))
        res[name] = {"input_bytes": int(zbuf.numel()), "inflate_ms_median": ms, "inflate_ms_all": times,
                     "output_gb_s": out_bytes / ms / 1e6, "segments_per_plane_mean": float(seg.mean()),
                     "segments_per_plane_max": int(seg.max()), "output_equal": ok}
    return res


def decompress_leg(reps):
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    from aeaj.codec import get_codec
    imgs = [Image.from_uint8(fr, ".png") for fr in bench.frames_u8(range(8), 1080, 1920, os.cpu_count() or 1)]
    st = JpegCompressionSettings("YCoCg", (40, 80), (4, 64))
    files = {"zlib9_files": Jpeg(st).compress_batch(imgs), "device_coded_files": Jpeg(st, deflate="device").compress_batch(imgs)}
    readers = {"host": Jpeg(st), "device": Jpeg(st, deflate="device")}
    mp = len(imgs) * 1080 * 1920 / 1e6
    res = {"workload": "8 synthetic 1920x1080 frames, YCoCg q40-80 b4-64, Jpeg.decompress_batch incl. .ajpg parsing, wall clock, "
                       "host / device alternated", "host_threads": os.cpu_count()}
    for fk, blobs in files.items():
        for j in readers.values():
            j.decompress_batch(blobs[:2])
            j.decompress_batch(blobs)
        r = {k: [] for k in readers}
        outs = {}
        for _ in range(reps):
            for k, j in readers.items():
                t0 = time.perf_counter()
                outs[k] = j.decompress_batch(blobs)
                r[k].append(mp / (time.perf_counter() - t0))
        res[fk] = {"bytes": int(sum(map(len, blobs))), **{f"{k}_mp_s": v for k, v in r.items()},
                   **{f"{k}_mp_s_median": float(np.median(v)) for k, v in r.items()},
                   "speedup": float(np.median(r["device"]) / np.median(r["host"])),
                   "decoded_equal": all(np.array_equal(a.data, b_.data) for a, b_ in zip(outs["host"], outs["device"]))}
    # where the host path's time goes, on the zlib-9 files: framing + zlib, the int32 upload, the device decode
    j = readers["host"]
    codec = get_codec()
    blobs = files["zlib9_files"]
    t = {"parse_and_zlib_s": [], "upload_s": [], "device_s": []}
    for _ in range(reps):
        t0 = time.perf_counter()
        parsed = [j._entropy_decode(x) for x in blobs]
        t1 = time.perf_counter()
        p0 = parsed[0]
        coef, leaves, counts = codec.upload_for_decode([p["layers"] for p in parsed], len(parsed), p0["H"], p0["W"], p0["space"],
                                                       p0["quality"], p0["blocks"])
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        codec.decode(coef, leaves, counts, len(parsed), p0["H"], p0["W"], p0["space"], p0["quality"], p0["blocks"], zigzag=True).cpu()
        t3 = time.perf_counter()
        t["parse_and_zlib_s"].append(t1 - t0); t["upload_s"].append(t2 - t1); t["device_s"].append(t3 - t2)
    res["host_path_breakdown_zlib9_files"] = {k: float(np.median(v)) for k, v in t.items()}
    res["host_path_breakdown_zlib9_files"]["int32_bytes_uploaded"] = int(sum(4 * len(L["coef"]) for p in parsed for L in p["layers"]))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the result to this file")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--legs", default="deflate,inflate", help="comma-separated: deflate, inflate")
    args = ap.parse_args()
    legs = set(args.legs.split(","))
    if not torch.cuda.is_available():
        raise SystemExit("deflate_bench needs a CUDA device")
    from aeaj.codec import get_codec
    codec = get_codec(0)
    res = {"gpu": card()}
    if "deflate" in legs:
        res.update(kernel=kernel_leg(codec, 3 * args.reps), compress_full=compress_leg(args.reps))
    if "inflate" in legs:
        res.update(inflate_kernel=inflate_kernel_leg(codec, 3 * args.reps), decompress_full=decompress_leg(args.reps))
    print(json.dumps(res), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
