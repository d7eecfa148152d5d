"""GPU tests of the device zlib decoder (aeaj_inflate_coefficients, Jpeg(deflate="device").decompress*): the CPU corpus of
test_inflate_cpu through the C ABI -- the same status and segment count as the host build of csrc/inflate_core.h, zlib's
bytes, nothing written past the expected length -- plus neighbouring streams, concurrent streams, CUDA-graph capture, and
every golden .ajpg file decoded bit-identically to the host path.  Run on the B200 box:  pytest tests -m gpu"""
import io
import json
import zlib

import numpy as np
import pytest

from test_deflate_cpu import build_checker as build_deflate_checker
from test_inflate_cpu import (BIG, LENGTH, OK, TRUNCATED, build_checker, corpus, host_inflate, mutations, payload,
                              zlib_verdict)
from test_device_deflate import _golden_names

pytestmark = pytest.mark.gpu

SPACE, Q, BR = "YCbCr", (50, 90), (4, 64)
B, H, W = 4, 1024, 1024                         # luma planes of 4 MiB, chroma of 1 MiB
CANARY = 0x5A


@pytest.fixture(scope="module")
def codec():
    from aeaj.codec import get_codec
    return get_codec(0)


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    return build_checker(tmp_path_factory.mktemp("inflate_gpu"))


@pytest.fixture(scope="module")
def exe_deflate(tmp_path_factory):
    return build_deflate_checker(tmp_path_factory.mktemp("inflate_gpu_deflate"))


def run_batch(codec, planes, instance=0, zbuf_extra=b""):
    """planes: {(b, l): (zlib bytes, expected bytes)} -> per plane (status, out_bytes, segments, output bytes, canary ok);
    streams are packed back to back in one input buffer"""
    import torch
    p = codec._plan(B, H, W, SPACE, BR, Q, instance)
    caps = [int(p.info.cap_coef[l]) for l in range(3)]
    blob, offs, lens = b"", np.zeros((B, 3), np.int64), np.zeros((B, 3), np.int64)
    counts = np.zeros((B, 3, 4), np.int32)
    for (b, l), (z, n) in planes.items():
        offs[b, l], lens[b, l] = len(blob), len(z)
        counts[b, l, 2] = n // 4
        blob += z
    blob += zbuf_extra
    dev = torch.device("cuda")
    zbuf = torch.from_numpy(np.frombuffer(blob, np.uint8).copy()).to(dev) if blob else torch.empty(0, dtype=torch.uint8, device=dev)
    for l in range(3):
        p.out.coef[l].view(torch.uint8).fill_(CANARY)
    ib = codec.inflate(zbuf, torch.from_numpy(offs).to(dev), torch.from_numpy(lens).to(dev), torch.from_numpy(counts).to(dev),
                       B, H, W, SPACE, Q, BR, instance=instance)
    torch.cuda.synchronize()
    st, ob, sg = ib.status.cpu().numpy(), ib.out_bytes.cpu().numpy(), ib.segments.cpu().numpy()
    res = {}
    for (b, l), (z, n) in planes.items():
        raw = ib.coef[l][b].view(torch.uint8).cpu().numpy()
        res[(b, l)] = (int(st[b, l]), int(ob[b, l]), int(sg[b, l]), raw[:min(n, 4 * caps[l])].tobytes(),
                       bool((raw[n:] == CANARY).all()))
    return res, caps


def check_corpus(codec, exe, tmp_path, streams):
    """every stream (payload a multiple of 4 bytes) through the device in mixed batches against the host build and zlib"""
    caps = [int(c) for c in codec._plan(B, H, W, SPACE, BR, Q).info.cap_coef]
    items = []
    for z in streams:
        st, data = zlib_verdict(z)
        if st == OK and len(data) % 4:
            continue
        items.append((z, len(data) if st == OK else min(BIG, 4 * caps[2]), data))
    host = host_inflate(exe, tmp_path, [(z, n) for z, n, _ in items])
    slots = [(b, l) for b in range(B) for l in range(3)]
    k = 0
    while k < len(items):
        planes, idx = {}, {}
        for (b, l) in slots:                                   # the next streams that fit, in mixed lengths
            if k < len(items) and items[k][1] <= 4 * caps[l]:
                planes[(b, l)] = items[k][:2]
                idx[(b, l)] = k
                k += 1
        assert planes, "a corpus stream does not fit any plane"
        got, _ = run_batch(codec, planes)
        for key, i in idx.items():
            z, n, data = items[i]
            st, ob, sg, out, canary = got[key]
            hst, hob, hsg, hout = host[i]
            assert (st, ob, sg) == (hst, hob, hsg), (i, z[:24].hex(), (st, ob, sg), (hst, hob, hsg))
            assert canary, (i, "written past the expected length")
            if data is not None:
                assert st == OK and out == data, i
    return host


def test_corpus_through_the_abi(codec, exe, exe_deflate, tmp_path):
    cases = corpus(exe_deflate, tmp_path)
    host = check_corpus(codec, exe, tmp_path, list(cases.values()))
    print(f"[inflate] {len(cases)} corpus streams, segments {sorted({h[2] for h in host})}")


def test_golden_streams_through_the_abi(codec, exe, exe_deflate, tmp_path):
    from test_deflate_cpu import golden_layer_streams, host_deflate
    raws = golden_layer_streams()
    check_corpus(codec, exe, tmp_path, [zlib.compress(r, 9) for r in raws] + host_deflate(exe_deflate, tmp_path, raws))


def test_mutation_corpus_through_the_abi(codec, exe, exe_deflate, tmp_path):
    from test_inflate_cpu import flushed, stored_stream
    from test_deflate_cpu import host_deflate
    rng = np.random.default_rng(9)
    small = payload(rng, 120, density=0.5)
    seeds = [zlib.compress(small, 9), flushed(small, 3, zlib.Z_SYNC_FLUSH), stored_stream(small[:64]),
             host_deflate(exe_deflate, tmp_path, [small])[0]]
    check_corpus(codec, exe, tmp_path, [m for s in seeds for m in mutations(s, rng, edits=100)])


def test_neighbour_does_not_complete_a_truncated_stream(codec):
    raw = payload(np.random.default_rng(3), 40000)
    z = zlib.compress(raw, 6)
    planes = {(0, 0): (z[:-7], len(raw)), (0, 1): (z, len(raw)), (1, 0): (z[:len(z) // 2], len(raw))}
    got, _ = run_batch(codec, planes, zbuf_extra=z)
    assert got[(0, 0)][0] == TRUNCATED and got[(1, 0)][0] == TRUNCATED
    assert got[(0, 1)][0] == OK and got[(0, 1)][3] == raw
    assert all(g[4] for g in got.values())


def test_length_mismatch(codec):
    raw = payload(np.random.default_rng(5), 5000)
    z = zlib.compress(raw)
    got, _ = run_batch(codec, {(0, 0): (z, len(raw) - 8), (0, 1): (z, len(raw) + 8), (1, 0): (z, len(raw))})
    assert got[(0, 0)][:2] == (LENGTH, len(raw) - 8) and got[(0, 0)][4]
    assert got[(0, 1)][:2] == (LENGTH, len(raw))
    assert got[(1, 0)][0] == OK


def _device_coded(exe_deflate, tmp_path, n=6):
    from test_deflate_cpu import host_deflate
    rng = np.random.default_rng(13)
    raws = [payload(rng, int(k)) for k in rng.integers(20000, 200000, n)]
    return raws, host_deflate(exe_deflate, tmp_path, raws)


def test_two_streams_two_plans(codec, exe_deflate, tmp_path):
    import torch
    raws, zs = _device_coded(exe_deflate, tmp_path)
    planes = [{(b, 0): (zs[3 * k + b], len(raws[3 * k + b])) for b in range(3)} for k in range(2)]
    ref = [run_batch(codec, pl, instance=400 + k)[0] for k, pl in enumerate(planes)]
    p = [codec._plan(B, H, W, SPACE, BR, Q, 400 + k) for k in range(2)]
    s = [torch.cuda.Stream(), torch.cuda.Stream()]
    for t in p:
        for l in range(3):
            t.out.coef[l].view(torch.uint8).fill_(CANARY)
    torch.cuda.synchronize()
    outs = []
    for k in range(2):
        blob = b"".join(z for z, _ in planes[k].values())
        offs, lens, counts = np.zeros((B, 3), np.int64), np.zeros((B, 3), np.int64), np.zeros((B, 3, 4), np.int32)
        o = 0
        for (b, l), (z, n) in planes[k].items():
            offs[b, l], lens[b, l], counts[b, l, 2] = o, len(z), n // 4
            o += len(z)
        with torch.cuda.stream(s[k]):
            args = [torch.from_numpy(a).cuda() for a in (np.frombuffer(blob, np.uint8).copy(), offs, lens, counts)]
            outs.append((codec.inflate(*args, B, H, W, SPACE, Q, BR, instance=400 + k), args))
    torch.cuda.synchronize()
    for k in range(2):
        ib = outs[k][0]
        for (b, l), (z, n) in planes[k].items():
            assert int(ib.status[b, l]) == OK
            assert ib.coef[l][b].view(torch.uint8)[:n].cpu().numpy().tobytes() == raws[3 * k + b]
            assert int(ib.segments[b, l]) == ref[k][(b, l)][2] == -(-n // 65536)


def test_cuda_graph_of_inflate(codec, exe_deflate, tmp_path):
    import torch
    raws, zs = _device_coded(exe_deflate, tmp_path, 3)
    offs = np.zeros((B, 3), np.int64)
    lens = np.zeros((B, 3), np.int64)
    counts = np.zeros((B, 3, 4), np.int32)
    o = 0
    for b in range(3):
        offs[b, 0], lens[b, 0], counts[b, 0, 2] = o, len(zs[b]), len(raws[b]) // 4
        o += len(zs[b])
    args = [torch.from_numpy(a).cuda() for a in (np.frombuffer(b"".join(zs), np.uint8).copy(), offs, lens, counts)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            ib = codec.inflate(*args, B, H, W, SPACE, Q, BR, instance=2200)
    torch.cuda.synchronize()
    eager = [ib.coef[0][b].view(torch.uint8)[:len(raws[b])].cpu().numpy().tobytes() for b in range(3)]
    assert eager == raws
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        ib = codec.inflate(*args, B, H, W, SPACE, Q, BR, instance=2200)
    ib.coef[0].zero_()
    ib.status.fill_(-1)
    g.replay()
    torch.cuda.synchronize()
    assert [ib.coef[0][b].view(torch.uint8)[:len(raws[b])].cpu().numpy().tobytes() for b in range(3)] == eager
    assert (ib.status[:3, 0] == 0).all()


def _load_ajpg(name):
    import os
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    for f in ("golden.npz", "golden_natural.npz"):
        z = np.load(os.path.join(d, f))
        if name + "/ajpg" in z.files:
            return z[name + "/ajpg"].tobytes()
    raise KeyError(name)


def test_golden_files_decode_identically(golden):
    """the reference's 39 zlib-9 .ajpg files and their device-coded counterparts: decompress / decompress_uint8 /
    decompress_batch with the device inflate are bit-identical to the host path"""
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    names = _golden_names()
    assert len(names) == 39
    files = [_load_ajpg(n) for n in names]
    for name, data in zip(names, files):
        c = golden.case(name)
        st = JpegCompressionSettings(c["space"], tuple(c["quality"]), tuple(c["blocks"]))
        dev_file = Jpeg(st, deflate="device").compress(Image.from_array(golden.input_f32(name).copy(), None, ".png"))
        for blob in (data, dev_file):
            a = Jpeg(st).decompress(blob)
            b = Jpeg(st, deflate="device").decompress(blob)
            assert np.array_equal(a.data, b.data) and a.original_shape == b.original_shape, name
            assert np.array_equal(Jpeg(st).decompress_uint8(blob), Jpeg(st, deflate="device").decompress_uint8(blob)), name
    st = JpegCompressionSettings()
    host = Jpeg(st).decompress_batch(files)
    dev = Jpeg(st, deflate="device").decompress_batch(files)
    for a, b in zip(host, dev):
        assert np.array_equal(a.data, b.data)


def _sections(blob):
    s = io.BytesIO(blob)
    ml = int.from_bytes(s.read(4), "big")
    meta = json.loads(s.read(ml))
    pos = 4 + ml
    zs = []
    for _ in range(meta["num_layers"]):
        nbits = int.from_bytes(blob[pos:pos + 4], "big")
        pos += 8 + (nbits + 7) // 8
        zl = int.from_bytes(blob[pos:pos + 4], "big")
        zs.append((pos, zl))
        pos += 4 + zl
    return zs


def test_errors_match_the_host_path():
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    from synth import synth
    st = JpegCompressionSettings("YCbCr", (40, 80), (4, 64))
    good = Jpeg(st).compress(Image.from_array(synth(96, 160, seed=4), None, ".png"))
    (p0, zl0), (p1, zl1), _ = _sections(good)
    # a truncated zlib section: the length field shortened, the rest of the file shifted
    cut = 6
    trunc = good[:p0] + (zl0 - cut).to_bytes(4, "big") + good[p0 + 4:p0 + 4 + zl0 - cut] + good[p0 + 4 + zl0:]
    for j in (Jpeg(st), Jpeg(st, deflate="device")):
        with pytest.raises(zlib.error):
            j.decompress(trunc)
    # a valid zlib section of the wrong length
    raw = zlib.decompress(good[p1 + 4:p1 + 4 + zl1])
    z = zlib.compress(raw + bytes(8), 9)
    longer = good[:p1] + len(z).to_bytes(4, "big") + z + good[p1 + 4 + zl1:]
    for j in (Jpeg(st), Jpeg(st, deflate="device")):
        with pytest.raises(ValueError):
            j.decompress(longer)
    # the crafted headers of test_corrupt_streams_raise
    ml = int.from_bytes(good[:4], "big")
    meta = json.loads(good[4:4 + ml])
    body = good[4 + ml:]

    def with_meta(**kw):
        m = dict(meta)
        m.update(kw)
        mb = json.dumps(m).encode()
        return len(mb).to_bytes(4, "big") + mb + body
    patched = bytearray(good)
    patched[4 + ml + 4:4 + ml + 8] = (1024).to_bytes(4, "big")
    for bad in (with_meta(block_size_max=16), with_meta(height=48, width=80), with_meta(block_size_min=8), bytes(patched)):
        with pytest.raises(ValueError):
            Jpeg(JpegCompressionSettings(), deflate="device").decompress(bad)
