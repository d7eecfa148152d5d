"""for compute-sanitizer: small encode / decode runs through every kernel family (all size classes incl. the tcgen05 ones, stream
layout, packing, segment copies, the host pipeline, the halo-split schedule over emulated bands, a PQ space).
    compute-sanitizer --tool memcheck python tools/sanitize_small.py"""
import sys, torch, numpy as np
sys.path.insert(0, 'adaptive-edge-aware-jpeg_b200'); sys.path.insert(0, 'tests')
from aeaj.codec import get_codec
from aeaj.tiled import TiledCodec
from synth import synth
c = get_codec(0)
q = (30, 95)
for space, (H, W), b, mask in (("YCbCr", (384, 512), (4, 128), 0xf), ("JzAzBz", (270, 480), (4, 64), 0xa), ("YCoCg", (135, 241), (2, 32), 0x0),
                               ("OKLAB", (300, 260), (2, 256), 0xa)):
    c.tensor_dct = mask
    rgb = torch.from_numpy(np.stack([synth(H, W, s) for s in (1, 2)])).cuda()
    enc = c.encode(rgb, space, q, b, stream=True)
    dec = c.decode_encoded(enc, space, q, b)
    c.check_status(enc.status, "encode")
    enc = c.encode(rgb, space, q, b)
    pk = c.pack(enc, space, q, b)
    c.unpack(pk, 2, H, W, space, q, b)
    dec2 = c.decode_encoded(enc, space, q, b, out="u8")
    torch.cuda.synchronize()
c.tensor_dct = 0xa
fr = torch.from_numpy(np.stack([(synth(270, 480, s) * 255).astype(np.uint8) for s in range(4)])).pin_memory()
out = torch.empty_like(fr).pin_memory()
for packed in (True, False):
    c.roundtrip_host_pipelined(fr, out, "YCbCr", q, (4, 64), slots=3, lag=2, packed=packed)
rgb = torch.from_numpy(synth(1024, 640, 21)).cuda()
t = TiledCodec(c, emulate=2)
enc = t.encode(rgb, 1024, 640, "ICtCp", q, (4, 128))
t.decode(enc, 1024, 640, "ICtCp", q, (4, 128))
torch.cuda.synchronize()
print("sanitize_small ok")
