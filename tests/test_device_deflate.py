"""GPU tests of the device entropy coder (aeaj_deflate_coefficients, Jpeg(deflate="device")): every stream is a valid zlib
stream with the host path's payload, the bytes equal the sequential host build's (csrc/deflate_core.h), and they depend
only on the input.  Run on the B200 box:  pytest tests -m gpu"""
import json
import os
import zlib

import numpy as np
import pytest

from test_deflate_cpu import C, build_checker, host_deflate, stored_bound

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def codec():
    from aeaj.codec import get_codec
    return get_codec(0)


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    return build_checker(tmp_path_factory.mktemp("deflate_gpu"))


def _golden_names():
    """every case for which the reference wrote an .ajpg file"""
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    names = []
    for f in ("golden.npz", "golden_natural.npz"):
        names += [k[: -len("/ajpg")] for k in np.load(os.path.join(d, f)).files if k.endswith("/ajpg")]
    return sorted(names)


def _sections(data: bytes):
    """(metadata + state sections, [zlib streams]) of an .ajpg file"""
    import io
    s = io.BytesIO(data)
    head = [s.read(4)]
    head.append(s.read(int.from_bytes(head[0], "big")))
    meta = json.loads(head[1])
    zs = []
    for _ in range(meta["num_layers"]):
        a, b = s.read(4), s.read(4)
        head += [a, b, s.read((int.from_bytes(a, "big") + 7) // 8)]
        zs.append(s.read(int.from_bytes(s.read(4), "big")))
    assert not s.read()
    return b"".join(head), zs


def test_golden_cases_device_deflate(golden, codec, exe, tmp_path):
    """for every golden case: same payloads, headers, states and decoded pixels as the default path; the reference's own
    decoder (the oracle's) reads the device streams; the device bytes are the host build's"""
    import oracle as O
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    names = _golden_names()
    assert len(names) == 39
    total_dev = total_host = 0
    for name in names:
        c = golden.case(name)
        rgb = golden.input_f32(name)
        s = JpegCompressionSettings(c["space"], tuple(c["quality"]), tuple(c["blocks"]))
        host = Jpeg(s).compress(Image.from_array(rgb.copy(), None, ".png"))
        dev = Jpeg(s, deflate="device").compress(Image.from_array(rgb.copy(), None, ".png"))
        hh, hz = _sections(host)
        dh, dz = _sections(dev)
        assert hh == dh, (name, "header / state sections")
        raws = [zlib.decompress(z) for z in hz]
        assert [zlib.decompress(z) for z in dz] == raws, (name, "payloads")
        assert host_deflate(exe, tmp_path, raws) == dz, (name, "device bytes differ from the host build")
        for raw, z in zip(raws, dz):
            assert len(z) <= stored_bound(len(raw))
        total_dev += sum(map(len, dz))
        total_host += sum(map(len, hz))
        a, b = Jpeg(s).decompress(host), Jpeg(s).decompress(dev)
        assert np.array_equal(a.data, b.data), name
        assert np.array_equal(O.decompress(dev), O.decompress(host)), name
    print(f"[deflate] golden cases: device {total_dev} bytes, zlib-9 {total_host} bytes, ratio {total_dev / total_host:.4f}")


def _planes(codec, enc, df):
    """the used bytes of every plane's stream, per image"""
    import torch
    torch.cuda.synchronize()
    lengths = df.lengths.cpu().numpy()
    return [[df.out[l][i, :int(lengths[i, l])].cpu().numpy().tobytes() for l in range(3)] for i in range(enc.shape[0])]


def test_bytes_do_not_depend_on_batch_stream_or_repeat(codec):
    import torch
    from synth import synth
    space, q, b = "YCoCg", (40, 80), (4, 64)
    H, W = 288, 352
    imgs = torch.from_numpy(np.stack([synth(H, W, seed=40 + i) for i in range(4)])).cuda()
    enc4 = codec.encode(imgs, space, q, b, stream=True)
    four = _planes(codec, enc4, codec.deflate(enc4, space, q, b))
    again = _planes(codec, enc4, codec.deflate(enc4, space, q, b))
    assert four == again
    for i in range(4):
        enc1 = codec.encode(imgs[i:i + 1], space, q, b, stream=True)
        one = _planes(codec, enc1, codec.deflate(enc1, space, q, b))[0]
        assert one == four[i], i
    # two batches on two concurrent streams, two plan instances
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    s1.wait_stream(torch.cuda.current_stream()); s2.wait_stream(torch.cuda.current_stream())
    res = {}
    for k, (st, part) in enumerate(((s1, imgs[:2]), (s2, imgs[2:]))):
        with torch.cuda.stream(st):
            e = codec.encode(part, space, q, b, stream=True, instance=300 + k)
            res[k] = (e, codec.deflate(e, space, q, b, instance=300 + k))
    torch.cuda.synchronize()
    got = _planes(codec, *res[0]) + _planes(codec, *res[1])
    assert got == four


def test_crafted_streams_through_the_abi(codec, exe, tmp_path):
    """n = 0, chunk boundaries, multiples of the chunk, zeros and incompressible data, with counts written by hand"""
    import torch
    from aeaj.codec import EncodedBatch
    space, q, b = "YCbCr", (50, 90), (4, 64)
    H, W = 512, 512                                             # luma capacity 262144 coefficients = 16 chunks
    B = 4
    p = codec._plan(B, H, W, space, b, q)
    caps = [int(p.info.cap_coef[l]) for l in range(3)]
    rng = np.random.default_rng(5)
    wc = C // 4
    lens = [[0, 4, 1], [wc - 1, wc, wc + 1], [2 * wc, 3 * wc, caps[2]], [caps[0], caps[1] - 7, 17]]
    coef = [torch.zeros((B, caps[l]), dtype=torch.int32, device="cuda") for l in range(3)]
    counts = torch.zeros((B, 3, 4), dtype=torch.int32)
    raws = []
    for i in range(B):
        for l in range(3):
            n = lens[i][l]
            if i == 3 and l == 0:
                v = rng.integers(-2**31, 2**31, n, dtype=np.int64).astype(np.int32)                  # incompressible
            elif i == 2 and l == 2:
                v = np.zeros(n, np.int32)
            else:
                v = (rng.integers(-40, 40, n) * (rng.random(n) < 0.25)).astype(np.int32)
            coef[l][i, :n] = torch.from_numpy(v).cuda()
            coef[l][i, n:] = 12345                                                                   # never read
            counts[i, l, 2] = n
            raws.append(v.tobytes())
    enc = EncodedBatch(coef=coef, leaves=p.out.leaves, states=p.out.states, counts=counts.cuda(), status=p.out.status,
                       shape=(B, H, W))
    df = codec.deflate(enc, space, q, b)
    got = [z for img in _planes(codec, enc, df) for z in img]
    assert int(df.status[0]) == 0
    assert all(len(z) <= df.out[k % 3].shape[1] for k, z in enumerate(got))
    for raw, z in zip(raws, got):
        assert zlib.decompress(z) == raw
        assert len(z) <= stored_bound(len(raw))
    assert host_deflate(exe, tmp_path, raws) == got


def test_cuda_graph_of_encode_and_deflate(codec):
    import torch
    from synth import synth
    space, q, b = "YCoCg", (40, 80), (4, 64)
    rgb = torch.from_numpy(synth(272, 480, seed=21)).cuda().unsqueeze(0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            enc = codec.encode(rgb, space, q, b, stream=True, instance=2100)
            df = codec.deflate(enc, space, q, b, instance=2100)
    torch.cuda.synchronize()
    eager = _planes(codec, enc, df)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        enc = codec.encode(rgb, space, q, b, stream=True, instance=2100)
        df = codec.deflate(enc, space, q, b, instance=2100)
    for t in df.out:
        t.zero_()
    df.lengths.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert _planes(codec, enc, df) == eager
