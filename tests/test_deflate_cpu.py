"""CPU check of the chunked deflate coder (csrc/deflate_core.h, the sequential definition of what aeaj_deflate_coefficients
writes): tests/native/deflate_check.cpp builds it with g++, Python's zlib judges the streams it writes."""
import io
import json
import os
import subprocess
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C = 65536                                                  # DF_CHUNK


def build_checker(tmp_dir) -> str:
    exe = os.path.join(str(tmp_dir), "deflate_check")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "native", "deflate_check.cpp")])
    return exe


def host_deflate(exe, tmp_dir, blobs):
    """the host build's zlib stream of every byte string in `blobs`"""
    args = []
    for i, b in enumerate(blobs):
        src, dst = os.path.join(str(tmp_dir), f"in{i}.bin"), os.path.join(str(tmp_dir), f"out{i}.z")
        with open(src, "wb") as f:
            f.write(b)
        args += [src, dst]
    subprocess.check_call([exe, "streams"] + args, timeout=600)
    out = []
    for i in range(len(blobs)):
        with open(os.path.join(str(tmp_dir), f"out{i}.z"), "rb") as f:
            out.append(f.read())
    return out


def golden_layer_streams():
    """the 117 coefficient streams of the 39 golden .ajpg files the reference wrote, as the bytes it handed to zlib"""
    streams = []
    for f in ("golden.npz", "golden_natural.npz"):
        z = np.load(os.path.join(ROOT, "tests", "golden", f))
        for k in sorted(z.files):
            if not k.endswith("/ajpg"):
                continue
            s = io.BytesIO(z[k].tobytes())
            meta = json.loads(s.read(int.from_bytes(s.read(4), "big")))
            for _ in range(meta["num_layers"]):
                nbits = int.from_bytes(s.read(4), "big")
                s.read(4)
                s.read((nbits + 7) // 8)
                streams.append(zlib.decompress(s.read(int.from_bytes(s.read(4), "big"))))
    return streams


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    return build_checker(tmp_path_factory.mktemp("deflate"))


def stored_bound(n):
    """header + trailer + per chunk two stored-block headers and the sync-flush block"""
    return 6 + max(1, -(-n // C)) * 16 + n


def test_golden_corpus_round_trips_within_ratio(exe, tmp_path):
    streams = golden_layer_streams()
    assert len(streams) == 117
    got = host_deflate(exe, tmp_path, streams)
    for i, (raw, z) in enumerate(zip(streams, got)):
        assert zlib.decompress(z) == raw, i
        assert len(z) <= stored_bound(len(raw)), i
    ours, z9 = sum(map(len, got)), sum(len(zlib.compress(s, 9)) for s in streams)
    print(f"[deflate] golden corpus: {sum(map(len, streams))} bytes -> {ours} bytes, zlib-9 {z9} bytes, ratio {ours / z9:.4f}")
    assert ours <= 1.20 * z9


def de_bruijn(k, n):
    """every length-n word over k symbols exactly once (cyclic): no 4-byte string repeats when n = 4"""
    a, seq = [0] * k * n, []

    def db(t, p):
        if t > n:
            if n % p == 0:
                seq.extend(a[1:p + 1])
        else:
            a[t] = a[t - p]
            db(t + 1, p)
            for j in range(a[t - p] + 1, k):
                a[t] = j
                db(t + 1, t)
    db(1, 1)
    return bytes(seq)


def test_edge_inputs_round_trip(exe, tmp_path):
    rng = np.random.default_rng(3)
    smooth = (rng.integers(-3, 4, 3 * C) * (rng.random(3 * C) < 0.2)).astype(np.int32).tobytes()
    cases = {
        "empty": b"",
        "16 bytes": bytes(range(16)),
        "C - 1": smooth[:C - 1], "C": smooth[:C], "C + 1": smooth[:C + 1],
        "2 C": smooth[:2 * C], "3 C": smooth[:3 * C],
        "zeros": bytes(5 * C + 12),
        "random int32": rng.integers(-2**31, 2**31, 300_000 // 4, dtype=np.int64).astype(np.int32).tobytes(),
        "no repeats": de_bruijn(8, 4)[:4000],
        "one symbol, 1 byte": b"A", "one symbol": b"A" * 70_000,
    }
    got = dict(zip(cases, host_deflate(exe, tmp_path, list(cases.values()))))
    for name, raw in cases.items():
        z = got[name]
        assert zlib.decompress(z) == raw, name
        assert len(z) <= stored_bound(len(raw)), (name, len(z), len(raw))
        assert z[:2] == b"\x78\x9c" and int.from_bytes(z[-4:], "big") == zlib.adler32(raw), name
    assert got["empty"] == b"\x78\x9c\x03\x00" + (1).to_bytes(4, "big")          # one final fixed block holding only end-of-block
    assert len(got["zeros"]) < 2000
    rnd = cases["random int32"]
    assert len(got["random int32"]) <= len(rnd) + 6 + 16 * (-(-len(rnd) // C)), "incompressible input grows by the stored-block bound at most"
    # no 4-byte string repeats: no matches, a dynamic block over 8 literals that declares a single distance code
    z = got["no repeats"]
    first = z[2]
    assert first & 7 == 0b101, "one final dynamic-Huffman block"
    assert (first >> 3) + 257 <= 257 + 31 and ((z[3] >> 0) & 31) == 0, "HDIST = 1: one (unused) distance code"


def kraft(lens):
    return sum(2.0 ** -l for l in lens if l)


@pytest.mark.parametrize("maxbits,nsym", [(15, 286), (15, 30), (7, 19)])
def test_length_limiting_fibonacci(exe, maxbits, nsym):
    """Fibonacci frequencies give the deepest Huffman tree: lengths must be cut to the limit and the code stay complete"""
    fib = [1, 1]
    while len(fib) < nsym:
        fib.append(min(fib[-1] + fib[-2], 4_000_000))
    out = subprocess.run([exe, "lengths", str(maxbits)] + [str(f) for f in fib], capture_output=True, text=True, check=True)
    lens = [int(x) for x in out.stdout.split()]
    assert len(lens) == nsym and max(lens) == maxbits and min(lens) >= 1
    assert kraft(lens) == 1.0
    order = np.argsort(-np.array(fib), kind="stable")
    assert all(lens[order[i]] <= lens[order[i + 1]] for i in range(nsym - 1)), "a more frequent symbol never gets a longer code"


def test_degenerate_alphabets(exe):
    def lengths(maxbits, freqs):
        out = subprocess.run([exe, "lengths", str(maxbits)] + [str(f) for f in freqs], capture_output=True, text=True, check=True)
        return [int(x) for x in out.stdout.split()]
    assert lengths(15, [0, 0, 5, 0]) == [0, 0, 1, 0]               # one used symbol: a single 1-bit code
    assert lengths(15, [0, 3, 0, 9]) == [0, 1, 0, 1]
    assert lengths(15, [0] * 30) == [0] * 30
    assert kraft(lengths(7, [1] * 19)) == 1.0
