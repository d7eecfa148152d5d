"""measurement tool: the host-buffer pipeline (bench.py's e2e leg) over slots / lag, plus the pieces on their own:
pure copies through the same pinned buffers, and the device work of one frame.  usage: python tools/e2e_sweep.py [frames]"""
import sys, time, torch, numpy as np
sys.path.insert(0, 'adaptive-edge-aware-jpeg_b200'); sys.path.insert(0, 'tests')
from aeaj.codec import get_codec
from synth import synth
F = int(sys.argv[1]) if len(sys.argv) > 1 else 16
H, W = 2160, 3840
c = get_codec(0)
sp, q, b = 'YCbCr', (30, 95), (4, 128)
fr = np.stack([(synth(H, W, s) * 255).astype(np.uint8) for s in range(F)])
hin = torch.from_numpy(fr).pin_memory()
hout = torch.empty_like(hin).pin_memory()
mp = F * H * W / 1e6

def run(**kw):
    c.roundtrip_host_pipelined(hin, hout, sp, q, b, repeat=1, **kw)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    h2d, d2h = c.roundtrip_host_pipelined(hin, hout, sp, q, b, repeat=4, **kw)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / 4
    print(f"{kw}: {dt * 1e3 / F:.3f} ms/frame  {mp / dt:.0f} MP/s  {h2d / 4 / dt / 1e9:.1f} + {d2h / 4 / dt / 1e9:.1f} GB/s;  host blocked on the device "
          f"{c.pipeline_host_wait_s / 4 * 1e3 / F:.3f} ms/frame", flush=True)

for kw in (dict(slots=8, lag=3), dict(slots=12, lag=4), dict(slots=6, lag=2), dict(slots=16, lag=6)):
    run(**kw)

# pure copies of the same byte counts, both directions at once, 8 streams
streams = [torch.cuda.Stream() for _ in range(8)]
dbuf = [torch.empty((H, W, 3), dtype=torch.uint8, device='cuda') for _ in range(8)]
torch.cuda.synchronize()
t0 = time.perf_counter()
for rep in range(4):
    for f in range(F):
        s = streams[f % 8]
        with torch.cuda.stream(s):
            dbuf[f % 8].copy_(hin[f], non_blocking=True)
            hout[f].copy_(dbuf[f % 8], non_blocking=True)
torch.cuda.synchronize()
dt = (time.perf_counter() - t0) / 4
print(f"pixels only, H2D + D2H on 8 streams: {dt * 1e3 / F:.3f} ms/frame  {mp / dt:.0f} MP/s  {fr.nbytes / dt / 1e9:.1f} GB/s per direction")

# device work of one frame per stream, no copies
rgb = [torch.from_numpy(fr[f % F]).cuda() for f in range(8)]
for k in range(8):
    with torch.cuda.stream(streams[k]):
        e = c.encode(rgb[k].unsqueeze(0), sp, q, b, instance=k); pk = c.pack(e, sp, q, b, instance=k)
torch.cuda.synchronize()
t0 = time.perf_counter()
for rep in range(4):
    for f in range(F):
        k = f % 8
        with torch.cuda.stream(streams[k]):
            e = c.encode(rgb[k].unsqueeze(0), sp, q, b, instance=k)
            pk = c.pack(e, sp, q, b, instance=k)
            c.unpack(pk, 1, H, W, sp, q, b, instance=k)
            c.decode(e.coef, e.leaves, e.counts, 1, H, W, sp, q, b, instance=k, out="u8")
torch.cuda.synchronize()
dt = (time.perf_counter() - t0) / 4
print(f"device work only (encode + pack + unpack + decode, one frame per job, 8 streams): {dt * 1e3 / F:.3f} ms/frame  {mp / dt:.0f} MP/s")

# are copies of one direction served in issue order across streams?  H2D -> [kernel that does nothing for ~0.4 ms] -> D2H per job:
# with independent queues 8 streams hide the kernel completely (same 0.52 ms/frame); a FIFO would add it to every frame
for nstreams in (8, 16):
    streams = [torch.cuda.Stream() for _ in range(nstreams)]
    dbuf = [torch.empty((H, W, 3), dtype=torch.uint8, device='cuda') for _ in range(nstreams)]
    for cycles in (0, 800_000):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for rep in range(4):
            for f in range(F):
                k = f % nstreams
                with torch.cuda.stream(streams[k]):
                    dbuf[k].copy_(hin[f], non_blocking=True)
                    if cycles:
                        torch.cuda._sleep(cycles)
                    hout[f].copy_(dbuf[k], non_blocking=True)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 4
        print(f"H2D -> sleep({cycles} cycles) -> D2H on {nstreams} streams: {dt * 1e3 / F:.3f} ms/frame")
