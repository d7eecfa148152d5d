"""CPU check of the segment-parallel zlib decoder (csrc/inflate_core.h, the sequential definition of what
aeaj_inflate_coefficients gives): tests/native/inflate_check.cpp builds it with g++, and Python's zlib.decompress is the
judge -- the same accept / reject decision, the same bytes, the matching error category -- on the golden streams, the
device coder's streams, every zlib level x strategy x window, flushes, crafted headers and a mutation corpus."""
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from test_deflate_cpu import build_checker as build_deflate_checker, golden_layer_streams, host_deflate

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# statuses (csrc/inflate_core.h)
OK, HEADER, NEED_DICT, BLOCK_TYPE, STORED_LEN, CODE_LENGTHS, BAD_SYMBOL, DIST_FAR, TRUNCATED, CHECK, LENGTH = range(11)
BIG = 1 << 22                                   # expected length for streams zlib rejects: never reached by these inputs


def category(msg: str) -> int:
    """the status a zlib.error message corresponds to"""
    table = [("incorrect header check", HEADER), ("invalid window size", HEADER), ("unknown compression method", HEADER),
             ("Error 2 ", NEED_DICT), ("invalid block type", BLOCK_TYPE), ("invalid stored block lengths", STORED_LEN),
             ("too many length or distance symbols", CODE_LENGTHS), ("invalid code lengths set", CODE_LENGTHS),
             ("invalid bit length repeat", CODE_LENGTHS), ("invalid literal/lengths set", CODE_LENGTHS),
             ("invalid distances set", CODE_LENGTHS), ("missing end-of-block", CODE_LENGTHS),
             ("invalid literal/length code", BAD_SYMBOL), ("invalid distance code", BAD_SYMBOL),
             ("invalid distance too far back", DIST_FAR), ("incomplete or truncated stream", TRUNCATED),
             ("incorrect data check", CHECK)]
    for key, code in table:
        if key in msg:
            return code
    raise AssertionError(f"unmapped zlib error: {msg}")


def zlib_verdict(z: bytes):
    """(status, bytes): Python's zlib.decompress as the reference"""
    try:
        return OK, zlib.decompress(z)
    except zlib.error as e:
        return category(str(e)), None


def build_checker(tmp_dir) -> str:
    exe = os.path.join(str(tmp_dir), "inflate_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "native", "inflate_check.cpp")])
    return exe


def host_inflate(exe, tmp_dir, items):
    """items: [(zlib bytes, expected length)] -> [(status, bytes produced, merged segments, output or None)]"""
    src, dst = os.path.join(str(tmp_dir), "inflate_in.bin"), os.path.join(str(tmp_dir), "inflate_out.bin")
    with open(src, "wb") as f:
        for z, n in items:
            f.write(struct.pack("<QQ", len(z), n))
            f.write(z)
    subprocess.check_call([exe, src, dst], timeout=600)
    res = []
    with open(dst, "rb") as f:
        for _ in items:
            st, n, seg = struct.unpack("<iqi", f.read(16))
            res.append((st, n, seg, f.read(n) if st == OK else None))
    return res


def payload(rng, n_int32, density=0.2, span=40):
    """a coefficient-like int32 stream: mostly zeros, small values"""
    return (rng.integers(-span, span + 1, n_int32) * (rng.random(n_int32) < density)).astype(np.int32).tobytes()


def flushed(data: bytes, parts: int, mode, level=6) -> bytes:
    c = zlib.compressobj(level)
    step = -(-len(data) // parts)
    out = b""
    for k in range(parts):
        out += c.compress(data[k * step:(k + 1) * step])
        if k < parts - 1:
            out += c.flush(mode)
    return out + c.flush()


def stored_stream(data: bytes) -> bytes:
    """one final stored block"""
    return b"\x78\x01" + b"\x01" + struct.pack("<HH", len(data), len(data) ^ 0xffff) + data + zlib.adler32(data).to_bytes(4, "big")


def corpus(exe_deflate, tmp_dir):
    """named zlib streams of int32 payloads (lengths multiples of 4): every kind the decoder must read or reject"""
    rng = np.random.default_rng(11)
    cases = {}
    base = payload(rng, 3000)
    strategies = {"default": zlib.Z_DEFAULT_STRATEGY, "filtered": zlib.Z_FILTERED, "huffman": zlib.Z_HUFFMAN_ONLY,
                  "rle": zlib.Z_RLE, "fixed": zlib.Z_FIXED}
    for level in range(10):
        for sname, strat in strategies.items():
            for wbits in range(9, 16):
                c = zlib.compressobj(level, zlib.DEFLATED, wbits, 8, strat)
                cases[f"l{level}-{sname}-w{wbits}"] = c.compress(base) + c.flush()
    cases["empty"] = zlib.compress(b"")
    big = payload(rng, 150_000, density=0.1)
    cases["sync-flush x7"] = flushed(big, 8, zlib.Z_SYNC_FLUSH)
    cases["full-flush x7"] = flushed(big, 8, zlib.Z_FULL_FLUSH)
    cases["sync-flush back-to-back"] = flushed(big[:40000], 3, zlib.Z_SYNC_FLUSH) + b""
    rep = bytes(4) * 50 + b"\x00\x00\xff\xff" * 300 + payload(rng, 500)
    cases["stored with 00 00 ff ff"] = stored_stream(rep)
    cases["level 0 with 00 00 ff ff"] = zlib.compress(rep * 200, 0)
    dev_in = [payload(rng, n) for n in (0, 1, 16383, 16384, 16385, 60000)] + [bytes(4 * 70000)]
    for i, z in enumerate(host_deflate(exe_deflate, tmp_dir, dev_in)):
        cases[f"device coder {i}"] = z
    return cases


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    return build_checker(tmp_path_factory.mktemp("inflate"))


@pytest.fixture(scope="module")
def exe_deflate(tmp_path_factory):
    return build_deflate_checker(tmp_path_factory.mktemp("inflate_deflate"))


def check_against_zlib(exe, tmp_path, streams):
    """every stream: same decision, bytes and category as zlib.decompress; returns the host results"""
    verdicts = [zlib_verdict(z) for z in streams]
    items = [(z, len(v[1]) if v[0] == OK else BIG) for z, v in zip(streams, verdicts)]
    got = host_inflate(exe, tmp_path, items)
    for i, ((st, data), (gst, n, seg, out)) in enumerate(zip(verdicts, got)):
        assert gst == st, (i, streams[i][:32].hex(), st, gst)
        if st == OK:
            assert out == data, i
    return got


def test_golden_zlib9_streams(exe, tmp_path):
    raws = golden_layer_streams()
    zs = [zlib.compress(r, 9) for r in raws]
    assert len(zs) == 117
    got = check_against_zlib(exe, tmp_path, zs)
    assert all(seg == 1 for _, _, seg, _ in got), "zlib-9 streams have no sync points: one segment"


def test_device_coder_streams_one_segment_per_chunk(exe, exe_deflate, tmp_path):
    raws = golden_layer_streams()
    zs = host_deflate(exe_deflate, tmp_path, raws)
    got = check_against_zlib(exe, tmp_path, zs)
    for raw, (_, _, seg, _) in zip(raws, got):
        assert seg == max(1, -(-len(raw) // 65536))


def test_corpus(exe, exe_deflate, tmp_path):
    cases = corpus(exe_deflate, tmp_path)
    names = list(cases)
    got = dict(zip(names, check_against_zlib(exe, tmp_path, [cases[k] for k in names])))
    assert all(got[k][0] == OK for k in names), [k for k in names if got[k][0] != OK]
    assert got["full-flush x7"][2] == 8, "Z_FULL_FLUSH: flushes + 1 segments"
    assert got["sync-flush x7"][2] < 8, "Z_SYNC_FLUSH matches across flushes merge segments"
    assert got["empty"][2] == 1
    for k in names:
        if k.startswith("l") and "-w" in k:
            assert got[k][2] == 1, k
    assert got["device coder 6"][2] == 5


def test_headers(exe, tmp_path):
    raw = payload(np.random.default_rng(2), 500)
    z = zlib.compress(raw)
    body = z[2:]

    def hdr(cmf, flg_hi):
        v = (cmf << 8) | flg_hi
        return bytes([cmf, flg_hi + (31 - v % 31) % 31])
    variants = {
        "cinfo 8": hdr(0x88, 0x80) + body, "method 7": hdr(0x77, 0x80) + body, "bad fcheck": bytes([0x78, 0x9d]) + body,
        "fdict": hdr(0x78, 0xa0) + b"\x00\x00\x00\x01" + body, "fdict truncated": hdr(0x78, 0xa0) + b"\x00\x01",
        "trailing bytes": z + b"\x00\x00\xff\xffgarbage", "one byte": z[:1], "cinfo 0": hdr(0x08, 0x80) + body,
        "cinfo 7 level 0": hdr(0x78, 0x00) + body,
    }
    got = check_against_zlib(exe, tmp_path, list(variants.values()))
    st = dict(zip(variants, [g[0] for g in got]))
    assert st["cinfo 8"] == HEADER and st["method 7"] == HEADER and st["bad fcheck"] == HEADER
    assert st["fdict"] == NEED_DICT and st["fdict truncated"] == TRUNCATED
    assert st["trailing bytes"] == OK and st["one byte"] == TRUNCATED


def test_expected_length(exe, tmp_path):
    raw = payload(np.random.default_rng(4), 5000)
    z = zlib.compress(raw)
    got = host_inflate(exe, tmp_path, [(z, len(raw)), (z, len(raw) - 4), (z, len(raw) + 4), (z, 0)])
    assert [g[0] for g in got] == [OK, LENGTH, LENGTH, LENGTH]
    assert got[1][1] == len(raw) - 4, "stops at the expected length"
    assert got[2][1] == len(raw)


def mutations(z: bytes, rng, edits=200):
    out = [z[:k] for k in range(len(z))]
    out += [z[:i] + bytes([z[i] ^ (1 << b)]) + z[i + 1:] for i in range(len(z)) for b in range(8)]
    for _ in range(edits):
        m = bytearray(z)
        for _ in range(int(rng.integers(1, 4))):
            m[int(rng.integers(0, len(m)))] = int(rng.integers(0, 256))
        out.append(bytes(m))
    return out


def test_mutation_corpus(exe, exe_deflate, tmp_path):
    rng = np.random.default_rng(7)
    small = payload(rng, 120, density=0.5)
    seeds = [zlib.compress(small, 9), zlib.compress(small, 1), flushed(small, 3, zlib.Z_SYNC_FLUSH),
             zlib.compressobj(9, zlib.DEFLATED, 15, 8, zlib.Z_FIXED).compress(small) + b"", stored_stream(small[:64]),
             host_deflate(exe_deflate, tmp_path, [small])[0]]
    c = zlib.compressobj(9, zlib.DEFLATED, 15, 8, zlib.Z_FIXED)
    seeds[3] = c.compress(small) + c.flush()
    streams = [m for s in seeds for m in mutations(s, rng)]
    got = check_against_zlib(exe, tmp_path, streams)
    cats = {g[0] for g in got}
    print(f"[inflate] {len(streams)} mutated streams, statuses {sorted(cats)}")
    assert {OK, TRUNCATED, CHECK, HEADER, BAD_SYMBOL} <= cats
