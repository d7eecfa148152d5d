"""Real multi-GPU halo-split check (run under torchrun on N GPUs of one box):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tests/multi_gpu_halo.py

Every rank encodes/decodes only its band of ONE image, reading halo rows and partial histograms from its neighbours'
shared workspaces over NVLink (aeaj/tiled.py) and compares the result with the fused single-GPU path computed locally."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "adaptive-edge-aware-jpeg_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import numpy as np
import torch
import torch.distributed as dist

from aeaj.codec import get_codec
from aeaj.tiled import TiledCodec, band_of
from synth import synth


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    os.environ.setdefault("NCCL_DEBUG", "WARN")
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    H, W = (int(a) for a in (args[:2] if len(args) >= 2 else (2048, 2048)))
    q, b = (30, 95), (4, 128)
    codec = get_codec(local)
    img = synth(H, W, seed=4)
    out = {}
    for space in ("JzAzBz", "ICtCp", "YCbCr"):
        full = torch.from_numpy(img).cuda()
        eg = codec.encode(full, space, q, b, instance=4000)
        ref = codec.download(eg)[0]
        ref_dec = codec.decode(eg.coef, eg.leaves, eg.counts, 1, H, W, space, q, b, instance=4000)[0].clone()
        lo, hi = band_of(rank, world, H)
        band = full[lo:hi].contiguous()
        t = TiledCodec(codec, rank, world)
        enc = t.encode(band, H, W, space, q, b, exchange_coef=True)          # parity: the whole stream on every rank
        got = codec.download(enc)[0]
        ok = all(np.array_equal(got[l][k], ref[l][k]) for l in range(3) for k in ("states", "leaves", "coef"))
        for _ in range(2):
            enc = t.encode(band, H, W, space, q, b)
            dec = t.decode(enc, H, W, space, q, b)
        torch.cuda.synchronize(); dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            enc = t.encode(band, H, W, space, q, b)
            dec = t.decode(enc, H, W, space, q, b)
        e1.record(); torch.cuda.synchronize(); dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1) / 5], device="cuda", dtype=torch.float64)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        t.check(H, W, space, q, b)
        ok = ok and bool(torch.equal(dec[lo:hi], ref_dec[lo:hi]))
        flag = torch.tensor([int(ok)], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        # single-GPU time for the same image, for the scaling figure
        for _ in range(2):
            eg = codec.encode(full, space, q, b, instance=4000)
            codec.decode(eg.coef, eg.leaves, eg.counts, 1, H, W, space, q, b, instance=4000)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            eg = codec.encode(full, space, q, b, instance=4000)
            codec.decode(eg.coef, eg.leaves, eg.counts, 1, H, W, space, q, b, instance=4000)
        e1.record(); torch.cuda.synchronize()
        t.close()
        out[space] = {"identical_to_single_gpu": bool(flag.item()), "ms_halo_split": float(ms.item()), "ms_single_gpu": e0.elapsed_time(e1) / 5,
                      "mp_per_s_halo_split": H * W / 1e6 / (float(ms.item()) / 1e3)}
    if rank == 0:
        print(json.dumps({"halo_split": {"gpus": world, "image": [H, W], "results": out}}))
    dist.destroy_process_group()
    if not all(v["identical_to_single_gpu"] for v in out.values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
