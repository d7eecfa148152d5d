"""GPU parity tests: the CUDA path (through the C ABI) against the pinned CPU oracle and against the
golden fixtures produced by the real reference.  Bit-exact for integer / byte / index work; float
tolerances are written beside each assertion.  Run on the B200 box:  pytest tests -m gpu"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import oracle as O                                   # checker only
from synth import synth

SPACES = ["YCbCr", "YCoCg", "YCoCg-R", "OKLAB", "ICaCb", "ICtCp", "JzAzBz"]


@pytest.fixture(scope="module")
def st():
    from aeaj.codec import get_stages
    return get_stages(0)


@pytest.fixture(scope="module")
def codec():
    from aeaj.codec import get_codec
    return get_codec(0)


def bits_differ(a, b):
    return int((np.ascontiguousarray(a).view(np.uint32) != np.ascontiguousarray(b).view(np.uint32)).sum())


# ------------------------------------------------------------------------------------------------
# colour
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("space", SPACES)
def test_color_forward_vs_oracle_and_golden(st, golden, space):
    rng = np.random.default_rng(3)
    rgb = (rng.integers(0, 256, (200_003, 3)).astype(np.float32) / 255.0).astype(np.float32)
    got = st.color(space, rgb, inverse=False)
    want = O.color_forward(space, rgb)
    if space in ("YCbCr", "YCoCg", "YCoCg-R"):
        assert bits_differ(got, want) == 0
    else:
        # f64 pow on the device vs glibc: identical after rounding to f32 except ~1e-5 of samples
        assert bits_differ(got, want) <= 12, bits_differ(got, want)
        assert np.abs(got - want).max() <= 2e-7 * max(1.0, float(np.abs(want).max()))
    g_rgb, g_ref = golden.get("color", "rgb"), golden.get("color", f"fwd_{space}")
    gg = st.color(space, g_rgb, inverse=False)
    tol = 0 if space in ("YCbCr", "YCoCg", "YCoCg-R") else (4e-7 if space == "OKLAB" else 1e-8)
    assert np.abs(gg - g_ref).max() <= tol


@pytest.mark.parametrize("space", SPACES)
def test_color_inverse_vs_oracle_and_golden(st, golden, space):
    x = golden.get("color", f"inv_in_{space}")
    got = st.color(space, x, inverse=True)
    want = O.color_inverse(space, x)
    ref = golden.get("color", f"inv_{space}")
    if space in ("YCbCr", "YCoCg", "YCoCg-R"):
        assert bits_differ(got, want) == 0 and bits_differ(got, ref) == 0
    else:
        assert np.abs(got - want).max() <= 1e-6
        assert np.abs(got - ref).max() <= (2e-5 if space == "OKLAB" else 1e-6)


def test_color_non_8bit_input_takes_f64_path(st):
    rng = np.random.default_rng(5)
    rgb = rng.random((50_001, 3)).astype(np.float32)            # not k/255: bypasses the sRGB LUT
    for space in ("OKLAB", "ICtCp", "JzAzBz"):
        got, want = st.color(space, rgb, False), O.color_forward(space, rgb)
        assert np.abs(got - want).max() <= 2e-7 * max(1.0, float(np.abs(want).max()))


@pytest.mark.parametrize("space", SPACES)
def test_normalisation_bit_exact(st, space):
    rng = np.random.default_rng(9)
    x = (rng.random(100_000).astype(np.float32) - 0.3).astype(np.float32)
    for ch in range(3):
        assert bits_differ(st.normalize(space, ch, x, False), O.normalize(space, ch, x, False)) == 0
        assert bits_differ(st.normalize(space, ch, x * 100, True), O.normalize(space, ch, x * 100, True)) == 0


def test_empty_inputs(st):
    assert st.color("YCbCr", np.zeros((0, 3), np.float32), False).shape == (0, 3)


# ------------------------------------------------------------------------------------------------
# resampling
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape,ratio", [((64, 96), (2, 2)), ((64, 96), (1, 4)), ((135, 241), (2, 2)), ((135, 241), (1, 4)),
                                         ((453, 618), (2, 2)), ((7, 9), (2, 2)), ((5, 4), (1, 4))])
def test_downsample_area_bit_exact(st, shape, ratio):
    rng = np.random.default_rng(1)
    x = rng.random(shape).astype(np.float32)
    h, w = shape[0] // ratio[0], shape[1] // ratio[1]
    assert bits_differ(st.downsample(x, h, w), O.downsample(x, h, w)) == 0


@pytest.mark.parametrize("shape,ratio", [((32, 48), (2, 2)), ((64, 24), (1, 4)), ((67, 120), (2, 2)), ((135, 60), (1, 4))])
def test_resize_linear_bit_exact(st, shape, ratio):
    rng = np.random.default_rng(2)
    x = rng.random(shape).astype(np.float32)
    H, W = shape[0] * ratio[0] + (1 if shape[0] % 2 else 0), shape[1] * ratio[1] + (1 if shape[1] % 2 == 0 and ratio[1] == 4 else 0)
    assert bits_differ(st.resize_linear(x, H, W), O.resize_linear(x, H, W)) == 0


# ------------------------------------------------------------------------------------------------
# Canny pipeline, stage-isolated (oracle inputs) and chained
# ------------------------------------------------------------------------------------------------
def _planes():
    rng = np.random.default_rng(4)
    out = [(synth(144, 256, seed=2)[..., 1] * 255).astype(np.uint8),
           (synth(135, 241, seed=3)[..., 0] * 255).astype(np.uint8),
           rng.integers(0, 256, (33, 17), dtype=np.uint8), rng.integers(0, 256, (4, 4), dtype=np.uint8),
           rng.integers(0, 5, (70, 130), dtype=np.uint8),                       # few-level plane (JzAzBz-like luma)
           rng.integers(0, 256, (1, 37), dtype=np.uint8), rng.integers(0, 256, (3, 2), dtype=np.uint8),
           np.full((40, 50), 77, dtype=np.uint8)]
    return out


def test_cast_u8_wraps_negative(st):
    x = np.array([[-0.19, 0.0, 0.5, 1.0, 1.2, -1.5, 0.999999]], dtype=np.float32)
    assert np.array_equal(st.cast_u8(x), O.cast_u8(x))
    rng = np.random.default_rng(0)
    y = (rng.random((50, 70)).astype(np.float32) * 3 - 1).astype(np.float32)
    assert np.array_equal(st.cast_u8(y), O.cast_u8(y))


@pytest.mark.parametrize("idx", range(8))
def test_canny_stages_bit_exact(st, idx):
    p = _planes()[idx]
    cl = O.clahe(p)
    assert np.array_equal(st.clahe(p), cl), "CLAHE"
    g = O.gauss3(cl)
    assert np.array_equal(st.gauss3(cl), g), "Gaussian"
    b = O.bilateral5(g)
    assert np.array_equal(st.bilateral5(g), b), "bilateral (f32 sequential fma model)"
    lo, hi = O.percentile_thresholds(b)
    assert st.percentile_thresholds(b) == (lo, hi), "percentile"
    assert np.array_equal(st.canny_u8(b, lo, hi), O.canny_u8(b, lo, hi)), "Canny + hysteresis"


def test_hysteresis_long_chains(st):
    """serpentine weak chain seeded by one strong pixel, crossing many tiles"""
    h, w = 300, 700
    img = np.zeros((h, w), dtype=np.uint8)
    for k, y in enumerate(range(10, h - 10, 12)):
        img[y:y + 3, 10:w - 10] = 120
        x = w - 13 if k % 2 == 0 else 10
        img[y:y + 15, x:x + 3] = 120
    img[10:13, 10:40] = 255
    for lo, hi in [(5.0, 200.0), (1.0, 100.0), (50.0, 60.0)]:
        assert np.array_equal(st.canny_u8(img, lo, hi), O.canny_u8(img, lo, hi))


@pytest.mark.parametrize("shape,seed", [((144, 256), 1), ((135, 241), 3), ((270, 480), 7), ((64, 64), 2)])
def test_canny_full_pipeline(st, shape, seed):
    rgb = synth(shape[0], shape[1], seed=seed)
    lay = O.color_forward("YCbCr", rgb.reshape(-1, 3)).reshape(shape[0], shape[1], 3)
    for c in range(3):
        layer = np.ascontiguousarray(lay[..., c])
        assert np.array_equal(st.canny(layer), O.canny(layer).astype(np.uint8))


# ------------------------------------------------------------------------------------------------
# quadtree
# ------------------------------------------------------------------------------------------------
QT_SHAPES = [(1, 1), (2, 2), (3, 5), (4, 4), (129, 1), (1, 129), (33, 17), (100, 100), (128, 128), (130, 257), (270, 480), (511, 513)]
QT_RANGES = [(4, 64), (4, 128), (2, 128), (8, 8), (16, 32), (4, 4), (64, 128), (2, 256), (32, 256)]


@pytest.mark.parametrize("shape", QT_SHAPES)
def test_quadtree_bit_exact(st, shape):
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    for density in (0.0, 0.002, 0.05, 1.0):
        edge = (rng.random(shape) < density).astype(np.float32)
        for (mn, mx) in QT_RANGES:
            if O.root_size(*shape) < mn or min(mx, O.root_size(*shape)) // mn > 128:
                continue
            leaves, states, root = st.quadtree(edge, mx, mn)
            wl, ws, wr = O.quadtree(edge, mx, mn)
            assert root == wr
            assert np.array_equal(states, ws), (shape, density, mn, mx, "states")
            assert np.array_equal(leaves[:, :3], wl), (shape, density, mn, mx, "leaves")
            off = np.concatenate([[0], np.cumsum(wl[:, 2].astype(np.int64) ** 2)])[:-1]
            assert np.array_equal(leaves[:, 3], off), "coefficient offsets"


# ------------------------------------------------------------------------------------------------
# DCT / quantiser
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("brange", [(4, 64), (4, 128), (2, 32), (8, 8), (64, 128), (16, 256)])
def test_dct_quant_and_inverse(st, brange):
    H, W = (200, 328) if brange[1] <= 128 else (300, 520)
    rgb = synth(H, W, seed=brange[1])
    layer = np.ascontiguousarray(O.color_forward("YCbCr", rgb.reshape(-1, 3)).reshape(H, W, 3)[..., 0])
    edge = O.canny(layer)
    leaves, states, root = O.quadtree(edge, brange[1], brange[0])
    assert len(set(leaves[:, 2].tolist())) >= 1
    for qrange in [(30, 95), (1, 99)]:
        tabs = O.qtables("YCbCr", qrange, brange)[0]
        mid, sc = O.NORM["YCbCr"]
        want, want_dct = O.encode_blocks(layer, "YCbCr", 0, leaves, tabs, want_dct=True)
        off = np.concatenate([[0], np.cumsum(leaves[:, 2].astype(np.int64) ** 2)])[:-1]
        lv4 = np.concatenate([leaves, off[:, None].astype(np.int32)], axis=1)
        got = st.dct_quant(layer, lv4, tabs, float(mid[0]), float(sc[0]), brange)
        d = got.astype(np.int64) - want.astype(np.int64)
        # T-DCT: f32 accumulation vs the oracle's f64 may flip exact .5 ties by one; none expected
        assert np.abs(d).max() <= 1 and int((d != 0).sum()) <= max(1, want.size // 100000), int((d != 0).sum())
        rec = st.dequant_idct(want, lv4, tabs, H, W, float(mid[0]), float(sc[0]), brange)
        ref = O.decode_blocks(want, leaves, tabs, H, W, "YCbCr", 0)
        assert np.abs(rec - ref).max() <= 2e-6            # f32 IDCT vs f64-accumulated oracle, values in [0,1]


def test_two_stage_calls_in_flight():
    """A stage call keeps its descriptors in its workspace: two aeaj_dct_quant calls on one handle, two workspaces and two
    streams, the first held back so that they overlap, give what each gives alone."""
    import ctypes as C
    import torch
    from aeaj import native
    lib, hd = native.load(), native.handle(0)
    H, W, brange = 200, 328, (4, 128)
    space = "YCbCr"
    layers = [np.ascontiguousarray(O.color_forward(space, synth(H, W, seed=s).reshape(-1, 3)).reshape(H, W, 3)[..., 0], dtype=np.float32)
              for s in (31, 32)]
    leaves, _, _ = O.quadtree(O.canny(layers[0]), brange[1], brange[0])       # one leaf list: the calls differ in their pixels only
    off = np.concatenate([[0], np.cumsum(leaves[:, 2].astype(np.int64) ** 2)])[:-1]
    n_coef = int((leaves[:, 2].astype(np.int64) ** 2).sum())
    lv = torch.from_numpy(np.ascontiguousarray(np.concatenate([leaves, off[:, None].astype(np.int32)], axis=1))).cuda()
    counts = torch.tensor([len(leaves), 0, n_coef, 0], dtype=torch.int32, device="cuda")
    tabs = O.qtables(space, (30, 95), brange)[0]
    tab_t = {s: torch.from_numpy(np.ascontiguousarray(m, dtype=np.int32)).cuda() for s, m in tabs.items()}
    qtab = (C.c_void_p * 9)()
    for s, t in tab_t.items():
        qtab[int(np.log2(s))] = t.data_ptr()
    mid, sc = O.NORM[space]
    src = [torch.from_numpy(l).cuda() for l in layers]
    ws = [torch.empty(int(lib.aeaj_stage_workspace_bytes(H, W, *brange)), dtype=torch.uint8, device="cuda") for _ in range(2)]
    out = [torch.empty(n_coef, dtype=torch.int32, device="cuda") for _ in range(2)]

    def call(k, stream):
        native.check(lib.aeaj_dct_quant(hd, src[k].data_ptr(), H, W, float(mid[0]), float(sc[0]), lv.data_ptr(), counts.data_ptr(),
                                        brange[0], brange[1], qtab, out[k].data_ptr(), ws[k].data_ptr(), stream.cuda_stream), "aeaj_dct_quant")

    alone = []
    for k in range(2):
        out[k].fill_(-1)
        call(k, torch.cuda.current_stream())
        torch.cuda.synchronize()
        alone.append(out[k].clone())
    assert not torch.equal(alone[0], alone[1])
    streams = [torch.cuda.Stream() for _ in range(2)]
    for s in streams:
        s.wait_stream(torch.cuda.current_stream())
    for o in out:
        o.fill_(-1)
    torch.cuda.synchronize()
    with torch.cuda.stream(streams[0]):
        torch.cuda._sleep(50_000_000)                      # the first call starts after the second one is enqueued and running
    call(0, streams[0])
    call(1, streams[1])
    torch.cuda.synchronize()
    for k in range(2):
        assert torch.equal(out[k], alone[k]), k


# ------------------------------------------------------------------------------------------------
# fused batch path + reference-facing shim
# ------------------------------------------------------------------------------------------------
def _check_layer(got_layer, ref_layer, coef_budget, tag):
    assert np.array_equal(got_layer["states"], ref_layer["states"]), f"{tag} states"
    assert np.array_equal(got_layer["leaves"][:, :3], ref_layer["leaves"]), f"{tag} leaves"
    assert got_layer["root"] == ref_layer["root"]
    d = np.abs(got_layer["coef"].astype(np.int64) - ref_layer["coef"].astype(np.int64))
    assert d.max() <= 1 and int((d != 0).sum()) <= coef_budget, (tag, int((d != 0).sum()))
    return int((d != 0).sum())


def _check_encode(layers, ref, coef_budget=2):
    for i in range(3):
        _check_layer(layers[i], ref[i], coef_budget, f"layer {i}")


EDGE_BUDGET_PX = 4        # per layer, PQ / cube-root spaces only (class T-POW: a 1-ULP colour difference flips a u8 truncation);
                          # the same budget test_oracle_golden.py gives the oracle against the reference


@pytest.mark.parametrize("space,shape,q,b", [("YCbCr", (144, 256), (30, 95), (4, 128)), ("YCoCg", (135, 241), (1, 99), (4, 64)),
                                             ("ICtCp", (96, 160), (40, 80), (4, 64)), ("ICaCb", (135, 241), (30, 95), (4, 32)),
                                             ("JzAzBz", (100, 100), (30, 95), (4, 128)), ("OKLAB", (64, 96), (50, 90), (2, 16)),
                                             ("YCoCg-R", (270, 480), (40, 80), (8, 64)),
                                             # BASELINE configs C5 (1080p, reference defaults, extreme quality) and C4's spaces at 2K
                                             ("YCoCg", (1080, 1920), (1, 99), (4, 64)), ("ICtCp", (1024, 2048), (30, 95), (4, 128)),
                                             ("JzAzBz", (1024, 1536), (30, 95), (4, 128)), ("OKLAB", (768, 1024), (30, 95), (4, 128)),
                                             # GUI-reachable extremes (main_frame.py:44-45): blocks 2 .. 256
                                             ("YCbCr", (300, 520), (30, 95), (2, 256)), ("YCoCg", (520, 300), (50, 90), (8, 256))])
def test_fused_encode_decode_vs_oracle(codec, space, shape, q, b):
    """Fused batch path against the oracle, layer by layer.  Linear spaces: layers and edge maps bit-exact, every quadtree
    equal.  PQ / cube-root spaces: at most EDGE_BUDGET_PX edge pixels may differ per layer (counted, never skipped), and
    every layer whose edge map matches must have the oracle's quadtree and coefficients."""
    import torch
    H, W = shape
    batch = np.stack([synth(H, W, seed=s) for s in (1, 2, 3)])
    enc = codec.encode(torch.from_numpy(batch).cuda(), space, q, b, taps=True)
    got = codec.download(enc)
    edges = [e.cpu().numpy() for e in enc.edges]
    lays = [l.cpu().numpy() for l in enc.layers]
    dec = codec.decode_encoded(enc, space, q, b).cpu().numpy()
    exact_color = space in ("YCbCr", "YCoCg", "YCoCg-R")
    n_layers = n_struct_equal = edge_px_total = coef_flips = 0
    for k in range(3):
        ref = O.encode_hot(batch[k], space, q, b)
        for i in range(3):
            if exact_color:
                assert bits_differ(lays[i][k], ref[i]["layer"]) == 0, "colour + downsample"
            else:
                assert np.abs(lays[i][k] - ref[i]["layer"]).max() <= 4e-7 * max(1.0, float(np.abs(ref[i]["layer"]).max()))
            mism = int((edges[i][k] != ref[i]["edge"].astype(np.uint8)).sum())
            assert mism <= (0 if exact_color else EDGE_BUDGET_PX), (space, k, i, "edge map mismatches", mism)
            n_layers += 1
            edge_px_total += mism
            if mism == 0:
                coef_flips += _check_layer(got[k][i], ref[i], 2 if exact_color else 50, f"{space} image {k} layer {i}")
                n_struct_equal += 1
        ref_dec = O.decode_hot([dict(leaves=got[k][i]["leaves"][:, :3], coef=got[k][i]["coef"]) for i in range(3)], H, W, space, q, b)
        lsb = np.abs((dec[k] * 255).astype(np.uint8).astype(int) - (ref_dec * 255).astype(np.uint8).astype(int))
        diff = np.abs(dec[k] - ref_dec)
        if space in ("ICaCb", "ICtCp", "JzAzBz"):
            # class T-NAN: near black, L'M'S' can come out a hair below zero; the reference's f64 pow then
            # yields NaN and its fastmath clamp turns the whole pixel white (1,1,1).  Which side of zero a
            # value lands on depends on the last bits of the IDCT, so such pixels are excluded (and bounded).
            nan_class = np.all(dec[k] == 1.0, axis=-1) | np.all(ref_dec == 1.0, axis=-1)
            assert nan_class.mean() < 2e-3
            lsb[nan_class] = 0
            diff[nan_class] = 0
        assert lsb.max() <= 1
        # float bound: 3e-6 for the linear spaces; in the PQ / cube-root spaces the inverse transfer function is steep near
        # black and amplifies the last-bit differences of an f32 IDCT (both the FP32 and the tensor-core kernels; the oracle
        # accumulates in f64) up to ~3e-5 on megapixel images -- the 8-bit bar above (<= 1 LSB) is the one that matters there
        assert diff.max() <= (5e-5 if space in ("ICaCb", "ICtCp", "JzAzBz", "OKLAB") else 3e-6)
    print(f"[parity] {space} {H}x{W}: quadtree+coefficients equal to the oracle's on {n_struct_equal}/{n_layers} layers, "
          f"{edge_px_total} edge px differ in total, {coef_flips} coefficient ties flipped")
    assert n_struct_equal >= n_layers - (0 if exact_color else 2)


def _golden_names():
    import json, os
    d = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    names = []
    for f in ("golden.json", "golden_natural.json"):
        with open(os.path.join(d, f)) as fh:
            names += [k for k, v in json.load(fh)["cases"].items() if v.get("mode") != "D"]
    return sorted(names)


@pytest.mark.parametrize("name", _golden_names())
def test_golden_reference_stream(golden, codec, name):
    """Jpeg.compress / decompress of the shim against the reference's own .ajpg stream (mode S), ONE named case at a time:
    byte identity where tests/golden/expected_parity.json pins it for the CUDA path, otherwise no more tie-class differences
    (edge pixels, coefficient flips) than pinned; lena, the synthetic cases, and the natural images of configuration C3
    (six odd-sized LIVE images + baboon + peppers in OKLAB) and one LIVE image per PQ space."""
    import parity_report as PR
    from pin_expected_parity import gpu_case
    from jpeg import Jpeg, JpegCompressionSettings
    c = golden.case(name)
    rgb = golden.input_f32(name)
    got = gpu_case(golden, name, codec)
    expected = PR.load_expected()
    exact = c["space"] in ("YCbCr", "YCoCg", "YCoCg-R")
    print(f"[parity] {name}: {'byte-identical' if got['byte_identical'] else 'differs'}", [(l["edge_px"], l["tree_equal"], l["coef_diffs"]) for l in got["layers"]])
    for i, l in enumerate(got["layers"]):
        assert l["edge_px"] <= (0 if exact else EDGE_BUDGET_PX), (name, i, "edge map")
        if l["edge_px"] == 0:
            assert l["tree_equal"], (name, i, "quadtree differs although the edge map matches")
        if l["tree_equal"]:
            assert l["coef_max_abs"] <= 1 and l["coef_diffs"] <= 8, (name, i, l)             # T-DCT: exact .5 ties only
    if "gpu" in expected:
        PR.check_against_expected("gpu", name, got, expected)
    ref_bytes = golden.get(name, "ajpg").tobytes()
    dec = Jpeg(JpegCompressionSettings()).decompress(ref_bytes)
    assert dec.data.shape == rgb.shape and dec.data.dtype == np.float32
    ref_u8 = golden.get(name, "decoded_u8_s3")
    lsb = np.abs(ref_u8.astype(int) - dec.get_uint8()[::3, ::3].astype(int))
    if c["space"] in ("ICaCb", "ICtCp", "JzAzBz"):
        # class T-NAN (DESIGN.md): near black a PQ-space L'M'S' value lands a hair on either side of zero depending on the
        # last bits of the IDCT; the reference's pow then returns NaN and its clamp paints the pixel white.  In flat black blocks
        # all pixels share one value, so a whole block flips together.  Counted and bounded by the size of the class itself.
        nan_class = np.all(ref_u8 == 255, axis=-1) | np.all(dec.get_uint8()[::3, ::3] == 255, axis=-1)
        differ = nan_class & (lsb.max(axis=-1) > 1)
        print(f"[parity] {name}: {int(differ.sum())} of {differ.size} sampled pixels are T-NAN flips")
        assert differ.mean() <= max(2.5 * nan_class.mean(), 1e-3), (name, float(differ.mean()), float(nan_class.mean()))
        lsb[nan_class] = 0
    assert lsb.max() <= 1, name


def test_pinned_gpu_identity_rate():
    import parity_report as PR
    exp = PR.load_expected()
    if "gpu" not in exp:
        pytest.skip("CUDA-path expectations not pinned yet (tests/golden/pin_expected_parity.py --gpu)")
    ident = [n for n, r in exp["gpu"].items() if r["byte_identical"]]
    print(f"[parity] {len(ident)} of {len(exp['gpu'])} reference streams reproduced byte for byte by the CUDA path")
    assert len(exp["gpu"]) == len(_golden_names()) and len(ident) >= 0.8 * len(exp["gpu"])


def test_corrupt_streams_raise(codec):
    """Crafted .ajpg headers (ADVICE r1): wrong root, leaves outside the block range, and -- through the C ABI directly -- leaf
    lists that do not fit the plan must be rejected / skipped, never written through."""
    import io, json, torch
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    rgb = synth(96, 160, seed=4)
    j = Jpeg(JpegCompressionSettings("YCbCr", (40, 80), (4, 64)))
    good = j.compress(Image.from_array(rgb, None, ".png"))
    ml = int.from_bytes(good[:4], "big")
    meta = json.loads(good[4:4 + ml])
    body = good[4 + ml:]
    def with_meta(**kw):
        m = dict(meta); m.update(kw)
        mb = json.dumps(m).encode()
        return len(mb).to_bytes(4, "big") + mb + body
    for bad in (with_meta(block_size_max=16),          # leaves of 32 / 64 are now outside the declared range
                with_meta(height=48, width=80),         # root no longer matches the layer
                with_meta(block_size_min=8)):           # 4 x 4 leaves below the declared minimum
        with pytest.raises(ValueError):
            Jpeg(JpegCompressionSettings()).decompress(bad)
    # root patched in the first layer header: bits_len(4) root(4)
    patched = bytearray(good)
    patched[4 + ml + 4:4 + ml + 8] = (1024).to_bytes(4, "big")
    with pytest.raises(ValueError):
        Jpeg(JpegCompressionSettings()).decompress(bytes(patched))
    # C ABI: a hostile leaf list (sizes 0, 3, 512, negative / far positions, wild offsets) is skipped and counted
    H, W, space, q, b = 192, 320, "YCbCr", (40, 80), (4, 64)
    enc = codec.encode(torch.from_numpy(synth(H, W, seed=4)).cuda(), space, q, b)
    lv = enc.leaves[0].clone()
    n = int(enc.counts[0, 0, 0])
    evil = torch.tensor([[0, 0, 0, 0], [4, 4, 3, 16], [0, 0, 512, 0], [-8, 0, 8, 0], [100000, 0, 8, 0], [0, 0, 8, 2 ** 30], [0, 0, 128, 0]],
                        dtype=torch.int32, device=lv.device)
    lv[0, :evil.shape[0]] = evil
    out = codec.decode([enc.coef[0], enc.coef[1], enc.coef[2]], [lv, enc.leaves[1], enc.leaves[2]], enc.counts, 1, H, W, space, q, b)
    torch.cuda.synchronize()
    assert int(codec.last_decode_status[3]) == evil.shape[0] and n > evil.shape[0]
    with pytest.raises(ValueError):
        codec.check_status(codec.last_decode_status, "decode")
    assert torch.isfinite(out).all()


def test_plan_cache_is_bounded():
    from aeaj.codec import DeviceCodec
    import torch
    c = DeviceCodec(0)
    c.MAX_PLANS = 3
    for k in range(6):
        H, W = 64 + 16 * k, 96
        enc = c.encode(torch.from_numpy(synth(H, W, seed=k)).cuda(), "YCbCr", (40, 80), (4, 64))
        dec = c.decode_encoded(enc, "YCbCr", (40, 80), (4, 64))
        assert dec.shape == (1, H, W, 3)
    assert len(c._plans) == 3
    c.close()
    assert len(c._plans) == 0


def _device_bytes(obj, seen):
    """bytes of the distinct CUDA tensors reachable from obj through dataclass fields, lists, tuples and dicts"""
    import dataclasses
    import torch
    if isinstance(obj, torch.Tensor):
        s = obj.untyped_storage()
        if not obj.is_cuda or s.data_ptr() in seen:
            return 0
        seen.add(s.data_ptr())
        return s.nbytes()
    if dataclasses.is_dataclass(obj):
        obj = [getattr(obj, f.name) for f in dataclasses.fields(obj)]
    elif isinstance(obj, dict):
        obj = list(obj.values())
    return sum(_device_bytes(v, seen) for v in obj) if isinstance(obj, (list, tuple)) else 0


def test_plan_bytes_count_every_buffer():
    """the plan-cache bound counts what a plan holds: after each call that allocates plan buffers on first use, every plan's
    nbytes equals the bytes of the device tensors it references"""
    from aeaj.codec import DeviceCodec
    import torch
    H, W, space, q, b = 136, 200, "YCbCr", (40, 80), (4, 64)
    c = DeviceCodec(0)

    def check(what):
        torch.cuda.synchronize()
        for key, p in c._plans.items():
            assert p.nbytes == _device_bytes(p, set()), (what, key, p.nbytes, _device_bytes(p, set()))

    rgb = torch.from_numpy(synth(H, W, seed=6)).cuda()
    enc = c.encode(rgb, space, q, b, stream=True)
    check("encode(stream=True)")
    for k in (1, 2, 4, 8):
        c.decode(enc.coef, enc.leaves, enc.counts, 1, H, W, space, q, b, zigzag=True, out="both", scale=k)
        check(f"decode(scale={k})")
    c.pack(enc, space, q, b)
    check("pack")
    df = c.deflate(enc, space, q, b)
    check("deflate")
    lengths = df.lengths.long()
    zbuf = torch.cat([df.out[l][0, :int(lengths[0, l])] for l in range(3)])
    offsets = torch.cumsum(lengths, 1) - lengths
    c.inflate(zbuf, offsets.contiguous(), lengths.contiguous(), enc.counts, 1, H, W, space, q, b)
    check("inflate")
    frames = torch.from_numpy(synth(H, W, seed=7)).unsqueeze(0).pin_memory()
    c.roundtrip_host_pipelined(frames, torch.empty_like(frames).pin_memory(), space, q, b, slots=2)
    check("roundtrip_host_pipelined")
    c.close()


def test_two_streams_with_256_leaves(codec):
    """ADVICE r1: the 256 x 256 kernel's intermediate tiles belong to the call -- two plans running concurrently on two
    streams (roundtrip_device) must not share them."""
    import torch
    H, W = 520, 784
    space, q, b = "YCbCr", (30, 95), (8, 256)
    frames = []
    for s in range(4):                                         # flat upper part (edge-free 256 x 256 blocks), textured lower part
        f = np.full((H, W, 3), np.float32(round((0.2 + 0.15 * s) * 255) / 255), np.float32)
        f[300:] = synth(H, W, seed=s)[300:]
        frames.append(f)
    batch = torch.from_numpy(np.stack(frames)).cuda()
    enc = codec.encode(batch, space, q, b)
    n256 = int(sum((codec.download(enc)[k][0]["leaves"][:, 2] == 256).sum() for k in range(4)))
    assert n256 >= 4                                           # the 256 class has work in every image
    one = codec.decode_encoded(enc, space, q, b).clone()
    for _ in range(3):
        parts = codec.roundtrip_device(batch, space, q, b, streams=2)
        torch.cuda.synchronize()
        assert torch.equal(torch.cat(parts), one)


def test_two_devices_one_process():
    """ADVICE r1: function attributes and occupancy are per device -- a second handle on another GPU in the same process."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from aeaj.codec import get_codec
    rgb = synth(272, 480, seed=3)
    outs = []
    for d in (0, 1):
        with torch.cuda.device(d):
            c = get_codec(d)
            enc = c.encode(torch.from_numpy(rgb).to(f"cuda:{d}"), "YCbCr", (30, 95), (4, 128))
            L = c.download(enc)[0]
            outs.append((L, c.decode_encoded(enc, "YCbCr", (30, 95), (4, 128)).cpu()))
    for i in range(3):
        for key in ("coef", "leaves", "states"):
            assert np.array_equal(outs[0][0][i][key], outs[1][0][i][key])
    assert torch.equal(outs[0][1], outs[1][1])


def test_shim_api_surface_and_errors():
    from color import apply_normalization, convert, get_color_spaces
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    from jpeg.edge_detection import EdgeDetection
    from jpeg.quadtree import QuadTree
    assert sorted(get_color_spaces()) == sorted(["ICaCb", "ICtCp", "JzAzBz", "OKLAB", "YCbCr", "YCoCg", "YCoCg-R"])
    with pytest.raises(ValueError):
        JpegCompressionSettings("nope")
    with pytest.raises(TypeError):
        Jpeg(JpegCompressionSettings()).compress(np.zeros((4, 4, 3), np.float32))
    with pytest.raises(TypeError):
        convert("sRGB", "YCbCr", [[0, 0, 0]])
    with pytest.raises(ValueError):
        convert("YCbCr", "OKLAB", np.zeros((2, 3), np.float32))
    with pytest.raises(ValueError):
        convert("sRGB", "YCbCr", np.zeros((2, 4), np.float32))
    with pytest.raises(TypeError):
        EdgeDetection.canny([[0.0]])
    with pytest.raises(ValueError):
        EdgeDetection.canny(np.zeros((2, 2, 2), np.float32))
    with pytest.raises(TypeError):
        QuadTree([[0.0]])
    rgb = synth(64, 96, seed=1)
    lay = convert("sRGB", "YCbCr", rgb.reshape(-1, 3))
    assert lay.shape == (64 * 96, 3) and lay.dtype == np.float32
    n = apply_normalization("YCbCr", lay, False)
    back = apply_normalization("YCbCr", n, True)
    assert np.abs(back - lay).max() < 1e-6
    edge = EdgeDetection.canny(np.ascontiguousarray(lay[:, 0].reshape(64, 96)))
    assert edge.dtype == np.float32 and set(np.unique(edge)) <= {0.0, 1.0}
    qt = QuadTree(edge, max_size=32, min_size=4)
    leaves, states = qt.get_leaves_and_states()
    wl, ws, wr = O.quadtree(edge, 32, 4)
    assert [(n.x, n.y, n.size) for n in leaves] == [tuple(r) for r in wl.tolist()]
    assert states == [("00", "01", "10")[s] for s in ws.tolist()]
    assert qt.root.size == wr and not qt.root.is_leaf()
    j = Jpeg(JpegCompressionSettings("YCbCr", (50, 90), (4, 64)))
    assert sorted(j.quantization_matrix_cache[0].keys()) == [4, 8, 16, 32, 64] and 64 in j.zigzag_cache
    out = Jpeg(JpegCompressionSettings()).decompress(j.compress(Image.from_array(rgb, None, ".png")))
    assert isinstance(out, Image) and out.extension == ".png" and out.data.min() >= 0 and out.data.max() <= 1


def test_full_size_properties(codec):
    """C2-sized run (3840x2160): size-independent properties -- leaves tile the layer exactly once,
    coefficient counts match, decode(encode(x)) is close to x, re-encoding is deterministic."""
    import torch
    H, W = 2160, 3840
    rgb = torch.from_numpy(synth(H, W, seed=0)).cuda()
    space, q, b = "YCbCr", (30, 95), (4, 128)
    enc = codec.encode(rgb, space, q, b)
    L = codec.download(enc)[0]
    shapes = O.layer_shapes(H, W, space)
    for i in range(3):
        lv = L[i]["leaves"]
        h, w = shapes[i]
        cover = np.zeros((h, w), dtype=np.int32)
        for x, y, s, _ in lv[:: max(1, len(lv) // 4000)]:
            cover[y:y + s, x:x + s] += 1
        assert cover.max() <= 1
        area = sum(int(min(s, h - y)) * int(min(s, w - x)) for x, y, s, _ in lv.tolist())
        assert area == h * w                                   # leaves tile the in-bounds area
        assert int((lv[:, 2].astype(np.int64) ** 2).sum()) == len(L[i]["coef"])
        assert np.array_equal(lv[:, 3], np.concatenate([[0], np.cumsum(lv[:, 2].astype(np.int64) ** 2)])[:-1])
        assert set(lv[:, 2].tolist()) <= {4, 8, 16, 32, 64, 128}
        sl, nc = __import__("aeaj.native", fromlist=["x"]).states_to_leaves(L[i]["states"], L[i]["root"], h, w)
        assert np.array_equal(sl, lv)                          # the state stream round-trips to the leaf list
    chk = [int(L[i]["coef"].astype(np.int64).sum()) for i in range(3)]
    dec = codec.decode_encoded(enc, space, q, b)
    mse = float(((dec[0] - rgb) ** 2).mean().item())
    assert 10 * np.log10(1.0 / mse) > 25.0
    # and, since the C oracle finishes a 4K frame in seconds, the full comparison at BASELINE's size
    ref = O.encode_hot(rgb.cpu().numpy(), space, q, b)
    _check_encode(L, ref, coef_budget=8)
    ref_dec = O.decode_hot(ref, H, W, space, q, b)
    got_dec = dec[0].cpu().numpy()
    assert np.abs((got_dec * 255).astype(np.uint8).astype(int) - (ref_dec * 255).astype(np.uint8).astype(int)).max() <= 1
    enc2 = codec.encode(rgb, space, q, b)
    L2 = codec.download(enc2)[0]
    assert chk == [int(L2[i]["coef"].astype(np.int64).sum()) for i in range(3)]


def test_tensor_core_dct_parity(codec):
    """The tcgen05 (3xTF32, TMEM) 128x128 DCT / IDCT kernels and the FP32-FMA kernels, both against the oracle on a 4K
    frame: the quantiser is exact in both, so coefficient differences are .5-tie flips of class T-DCT (|d| = 1); decoded
    samples stay within 1 LSB / 3e-6 of the oracle."""
    import torch
    H, W = 2160, 3840
    rgb = torch.from_numpy(synth(H, W, seed=5)).cuda()
    space, q, b = "YCbCr", (30, 95), (4, 128)
    ref = O.encode_hot(rgb.cpu().numpy(), space, q, b)
    ref_dec = O.decode_hot(ref, H, W, space, q, b)
    flips, err = {}, {}
    saved = codec.tensor_dct
    try:
        for mode in (False, True):
            codec.tensor_dct = mode
            enc = codec.encode(rgb, space, q, b)
            L = codec.download(enc)[0]
            assert not codec.tensor_dct_timed_out()
            n = 0
            for i in range(3):
                assert np.array_equal(L[i]["leaves"][:, :3], ref[i]["leaves"])
                d = np.abs(L[i]["coef"].astype(np.int64) - ref[i]["coef"].astype(np.int64))
                assert d.max() <= 1
                n += int((d != 0).sum())
            flips[mode] = n
            # decode the ORACLE's coefficients, so that the comparison isolates the inverse path
            lv4 = [np.concatenate([ref[i]["leaves"], np.concatenate([[0], np.cumsum(ref[i]["leaves"][:, 2].astype(np.int64) ** 2)])[:-1, None]],
                                  axis=1).astype(np.int32) for i in range(3)]
            up = codec.upload_for_decode([[dict(leaves=lv4[i], coef=ref[i]["coef"]) for i in range(3)]], 1, H, W, space, q, b)
            dec = codec.decode(*up, 1, H, W, space, q, b)[0].cpu().numpy()
            assert not codec.tensor_dct_timed_out()
            err[mode] = float(np.abs(dec - ref_dec).max())
            assert np.abs((dec * 255).astype(np.uint8).astype(int) - (ref_dec * 255).astype(np.uint8).astype(int)).max() <= 1
    finally:
        codec.tensor_dct = saved
    n128 = sum(int((ref[i]["leaves"][:, 2] == 128).sum()) for i in range(3))
    assert n128 > 100                                          # the tensor path actually had work
    print("T-DCT flips vs oracle: fp32 kernels", flips[False], " tensor-core 128x128", flips[True], " leaves128", n128,
          " decode max |err| vs oracle: fp32", err[False], " tensor", err[True])
    assert flips[False] <= 8 and flips[True] <= 8
    assert err[False] <= 3e-6 and err[True] <= 3e-6


@pytest.mark.parametrize("packed", [True, False])
@pytest.mark.parametrize("slots,lag", [(3, 2), (8, 3), (4, 3), (2, 1), (2, 3), (1, 2)])
def test_host_pipelined_roundtrip_matches_device_path(codec, slots, lag, packed):
    """the host-buffer API (bench.py's e2e leg) returns the same pixels as the device-resident path, whatever the number of
    stream slots (12 jobs: every slot is reused) and the lag, requested lags above slots - 1 included"""
    import torch
    H, W = 270, 480
    frames = np.stack([synth(H, W, seed=s) for s in range(6)])
    space, q, b = "YCbCr", (30, 95), (4, 64)
    host_in = torch.from_numpy(frames).pin_memory()
    host_out = torch.zeros_like(host_in).pin_memory()
    h2d, d2h = codec.roundtrip_host_pipelined(host_in, host_out, space, q, b, slots=slots, repeat=2, lag=lag, packed=packed)
    dev = codec.decode_encoded(codec.encode(host_in.cuda(), space, q, b), space, q, b).cpu()
    assert torch.equal(dev, host_out)
    assert h2d > 2 * frames.nbytes and d2h > 2 * frames.nbytes


@pytest.mark.parametrize("space,G,bmax", [("YCbCr", 1, 128), ("YCbCr", 2, 128), ("YCbCr", 4, 128), ("ICtCp", 2, 128), ("JzAzBz", 4, 128),
                                           ("YCbCr", 2, 256)])
def test_halo_split_bands_emulated_on_one_gpu(codec, space, G, bmax):
    """SURVEY 8e / config C4: the phase-wise, band-restricted pipeline (what each rank of a halo-split runs),
    emulated on one GPU as G bands over shared buffers, must reproduce the fused single-call result exactly."""
    import torch
    from aeaj.tiled import TiledCodec
    H, W = 1024, 640
    q, b = (30, 95), (4, bmax)
    rgb = torch.from_numpy(synth(H, W, seed=21)).cuda()
    ref = codec.download(codec.encode(rgb, space, q, b))[0]
    ref_dec = codec.decode_encoded(codec._plan(1, H, W, space, b, q).out, space, q, b)[0].clone()
    t = TiledCodec(codec, emulate=G)
    enc = t.encode(rgb, H, W, space, q, b)
    got = codec.download(enc)[0]
    for l in range(3):
        for k in ("states", "leaves", "coef"):
            assert np.array_equal(got[l][k], ref[l][k]), (space, G, l, k)
    dec = t.decode(enc, H, W, space, q, b)
    assert torch.equal(dec, ref_dec)


@pytest.mark.parametrize("space,shape,b", [("YCbCr", (200, 328), (4, 128)), ("YCoCg", (135, 241), (2, 32)), ("ICtCp", (96, 160), (8, 64))])
def test_device_stream_layout_matches_host_packing(codec, space, shape, b):
    """SURVEY 8f rank 1: zigzag-ordered coefficient blocks and the 2-bit state stream produced on the device are
    byte-identical to the host-side packing of the row-major result; decoding either layout gives the same pixels."""
    import torch
    H, W = shape
    q = (30, 95)
    rgb = torch.from_numpy(np.stack([synth(H, W, seed=s) for s in (3, 4)])).cuda()
    nat = codec.download(codec.encode(rgb, space, q, b))
    dec_nat = codec.decode_encoded(codec._plan(2, H, W, space, b, q).out, space, q, b).clone()
    enc = codec.encode(rgb, space, q, b, stream=True)
    zz = codec.download(enc)
    dec_zz = codec.decode_encoded(enc, space, q, b)
    assert torch.equal(dec_nat, dec_zz)
    for k in range(2):
        for l in range(3):
            assert np.array_equal(zz[k][l]["coef"], O.zigzag_stream(nat[k][l]["coef"], nat[k][l]["leaves"][:, :3]))
            assert zz[k][l]["packed_states"].tobytes() == O.pack_states(nat[k][l]["states"])
            assert np.array_equal(zz[k][l]["states"], nat[k][l]["states"])


@pytest.mark.parametrize("space,shape,b", [("YCbCr", (144, 256), (4, 128)), ("ICtCp", (96, 160), (4, 64)), ("YCoCg", (135, 241), (4, 64)),
                                             ("JzAzBz", (100, 100), (4, 128))])
def test_uint8_io_bit_exact(codec, space, shape, b):
    """8-bit pixels in (Image.load: astype(float32) / 255.0, image.py:84) and out (Image.get_uint8: (data * 255).astype(uint8),
    image.py:127): the u8 entry points give exactly what the float path gives on the converted data."""
    import torch
    H, W = shape
    q = (30, 95)
    px = np.stack([(synth(H, W, seed=s) * 255).astype(np.uint8) for s in (4, 9)])
    as_float = px.astype(np.float32) / 255.0
    ref = codec.download(codec.encode(torch.from_numpy(as_float).cuda(), space, q, b))
    enc = codec.encode(torch.from_numpy(px).cuda(), space, q, b)
    got = codec.download(enc)
    for k in range(2):
        for i in range(3):
            for key in ("coef", "leaves", "states"):
                assert np.array_equal(got[k][i][key], ref[k][i][key]), (k, i, key)
    f32, u8 = codec.decode_encoded(enc, space, q, b, out="both")
    f32, u8 = f32.cpu().numpy(), u8.cpu().numpy()
    assert np.array_equal(u8, (f32 * 255).astype(np.uint8))
    only = codec.decode_encoded(enc, space, q, b, out="u8").cpu().numpy()
    assert np.array_equal(only, u8)
    # the shim: an Image made from 8-bit pixels compresses to the same bytes as its float twin, decompress_uint8 == get_uint8
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    j = Jpeg(JpegCompressionSettings(space, q, b))
    img8 = Image.from_uint8(px[0], ".png")
    assert img8.uint8_source() is not None
    a = j.compress(img8)
    bb = j.compress(Image.from_array(as_float[0].copy(), None, ".png"))
    assert a == bb
    dec = Jpeg(JpegCompressionSettings()).decompress(a)
    assert np.array_equal(Jpeg(JpegCompressionSettings()).decompress_uint8(a), dec.get_uint8())
    _ = img8.data                                              # handing the floats out drops the shortcut
    assert img8.uint8_source() is None and np.array_equal(img8.data, as_float[0])


def test_packed_coefficient_streams(codec):
    """aeaj_pack_coefficients / aeaj_unpack_coefficients: the packed PCIe form is lossless, matches the host packer bit for
    bit, and flags values outside int16 instead of truncating them silently."""
    import torch
    from aeaj import native
    H, W = 270, 480
    space, q, b = "YCbCr", (30, 95), (4, 128)
    batch = torch.from_numpy(np.stack([synth(H, W, seed=s) for s in range(3)])).cuda()
    for stream in (False, True):                              # row-major and zigzag block layouts
        enc = codec.encode(batch, space, q, b, stream=stream)
        counts = enc.counts.cpu().numpy()
        want = [enc.coef[l].clone() for l in range(3)]
        pk = codec.pack(enc, space, q, b)
        pkc = pk.counts.cpu().numpy()
        for k in range(3):
            for l in range(3):
                n = int(counts[k, l, 2])
                ref = want[l][k, :n].cpu().numpy()
                nnz, n2, ovf, nw = (int(x) for x in pkc[k, l])
                assert (nnz, n2, ovf, nw) == (int((ref != 0).sum()), n, 0, (n + 31) // 32)
                m, v, _ = native.pack_coefficients_host(ref)
                assert np.array_equal(pk.mask[l][k, :nw].cpu().numpy().view(np.uint32), m)
                assert np.array_equal(pk.vals[l][k, :nnz].cpu().numpy(), v)
                assert np.array_equal(native.unpack_coefficients_host(m, v, n), ref)
        for l in range(3):
            enc.coef[l].fill_(-7)
        got = codec.unpack(pk, 3, H, W, space, q, b)
        for k in range(3):
            for l in range(3):
                n = int(counts[k, l, 2])
                assert torch.equal(got[l][k, :n], want[l][k, :n])
    enc.coef[1][2, 5] = 70000                                 # a value that does not fit 16 bits: that plane is flagged, others are not
    pkc = codec.pack(enc, space, q, b).counts.cpu().numpy()
    assert pkc[2, 1, 2] == 1 and pkc[:, 0, 2].sum() == 0 and pkc[0, 1, 2] == 0
    # the host-buffer pipeline: packed and raw int32 transport give the same pixels
    host_in = torch.from_numpy(np.stack([(synth(H, W, seed=s) * 255).astype(np.uint8) for s in range(5)])).pin_memory()
    a, c = torch.empty_like(host_in).pin_memory(), torch.empty_like(host_in).pin_memory()
    h1, d1 = codec.roundtrip_host_pipelined(host_in, a, space, q, b, slots=3, repeat=2, lag=2, packed=True)
    h2, d2 = codec.roundtrip_host_pipelined(host_in, c, space, q, b, slots=3, repeat=2, lag=2, packed=False)
    assert torch.equal(a, c) and h1 < 0.7 * h2 and d1 < 0.7 * d2


@pytest.fixture
def overflow_frames(codec):
    """codec.encode, wrapped: after the real call, the first coefficient of plane 0 becomes 65536 + k (k its value) in every
    call whose index modulo `period` is in `frames` -- a plane that does not fit int16, whose int16 truncation is k"""
    real = codec.encode
    sel = dict(frames=set(), period=1, calls=0)

    def encode(*args, **kw):
        enc = real(*args, **kw)
        if sel["calls"] % sel["period"] in sel["frames"]:
            enc.coef[0][0, :1] += 65536
        sel["calls"] += 1
        return enc

    codec.encode = encode
    try:
        yield sel
    finally:
        del codec.encode


def test_host_pipelined_int16_overflow_travels_as_int32(codec, overflow_frames):
    """a packed job in which a plane overflows int16 travels whole as raw int32 streams, the other jobs stay packed: the
    pixels are those of packed=False, the bytes lie between an all-packed and an all-int32 run"""
    import torch
    H, W = 270, 480
    space, q, b = "YCbCr", (30, 95), (4, 64)
    F = 5
    host_in = torch.from_numpy(np.stack([(synth(H, W, seed=s) * 255).astype(np.uint8) for s in range(F)])).pin_memory()
    clean, mixed, raw = (torch.empty_like(host_in).pin_memory() for _ in range(3))

    def run(out, packed):
        overflow_frames["calls"] = 0
        return codec.roundtrip_host_pipelined(host_in, out, space, q, b, slots=3, repeat=2, lag=2, packed=packed)

    h_pk, d_pk = run(clean, True)
    overflow_frames.update(frames={1, 3}, period=F)
    h_mix, d_mix = run(mixed, True)
    h_raw, d_raw = run(raw, False)
    assert torch.equal(mixed, raw)
    for f in range(F):                                         # the added 65536 reaches the pixels of the frames it was added to
        assert torch.equal(mixed[f], clean[f]) == (f not in (1, 3)), f
    assert h_pk < h_mix < h_raw and d_pk < d_mix < d_raw


def test_copy_segments_device_table(codec):
    """aeaj_copy_segments with more than the 64 ranges that travel in the kernel parameters: the table goes through the
    caller's device scratch.  80 ranges of mixed sizes and alignments gathered into one arena and scattered back, bit for
    bit; without the scratch table the call fails instead of launching."""
    import ctypes as C
    import torch
    from aeaj import native
    rng = np.random.default_rng(7)
    sizes = [0, 0, 1, 1, 2, 3, 4, 7, 15, 16, 17, 31, 32, 33, 64, 100, 255, 256, 4096, 65539, 300_000] + [int(n) for n in rng.integers(1, 5000, 59)]
    src_shift, arena_shift = (0, 4, 1, 8), (0, 4, 3)           # 16-byte, 4-byte and odd starts, in changing combinations
    spos = apos = 0
    ranges = []
    for i, n in enumerate(sizes):
        so, ao = spos + src_shift[i % 4], apos + arena_shift[i % 3]
        ranges.append((so, ao, n))
        spos, apos = (so + n + 31) & ~15, (ao + n + 31) & ~15
    src_h = rng.integers(0, 256, spos, dtype=np.uint8)
    src = torch.from_numpy(src_h).cuda()
    dst = torch.zeros_like(src)
    arena = torch.zeros(apos, dtype=torch.uint8, device="cuda")
    table = torch.empty(len(ranges) * C.sizeof(native.Segment), dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def segs(pairs):
        arr = (native.Segment * len(pairs))()
        for k, (s, d, n) in enumerate(pairs):
            arr[k].src, arr[k].dst, arr[k].bytes = s, d, n
        return arr

    gather = segs([(src.data_ptr() + so, arena.data_ptr() + ao, n) for so, ao, n in ranges] + [(None, None, 0)])
    scatter = segs([(arena.data_ptr() + ao, dst.data_ptr() + so, n) for so, ao, n in ranges])
    with pytest.raises(native.AeajError, match="more than 64 ranges"):
        native.check(codec.lib.aeaj_copy_segments(gather, len(gather), None, stream), "aeaj_copy_segments")
    native.check(codec.lib.aeaj_copy_segments(gather, len(gather), table.data_ptr(), stream), "aeaj_copy_segments")
    native.check(codec.lib.aeaj_copy_segments(scatter, len(scatter), table.data_ptr(), stream), "aeaj_copy_segments")
    want_arena, want_dst = np.zeros(apos, dtype=np.uint8), np.zeros(spos, dtype=np.uint8)
    for so, ao, n in ranges:
        want_arena[ao:ao + n] = src_h[so:so + n]
        want_dst[so:so + n] = src_h[so:so + n]
    assert np.array_equal(arena.cpu().numpy(), want_arena)
    assert np.array_equal(dst.cpu().numpy(), want_dst)


def test_cuda_graph_roundtrip_equals_eager(codec):
    """steady-state calls issue no host-to-device copy, so encode + decode can be captured into one CUDA graph"""
    import torch
    H, W = 272, 480
    space, q, b = "YCbCr", (30, 95), (4, 128)
    rgb = torch.from_numpy(synth(H, W, seed=8)).cuda().unsqueeze(0)
    eager = codec.decode_encoded(codec.encode(rgb, space, q, b), space, q, b).clone()
    g, res = codec.capture_roundtrip(rgb, space, q, b)
    for _ in range(3):
        res.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(res, eager)
    rgb.copy_(torch.from_numpy(synth(H, W, seed=9)).cuda())  # new pixels in the captured input buffer
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(res, codec.decode_encoded(codec.encode(rgb, space, q, b), space, q, b))


def test_cuda_graph_of_pack_and_unpack(codec):
    """steady-state pack / unpack issue no host-to-device copy either (the two keep separate descriptor tables): encode, pack,
    unpack and decode captured in one CUDA graph give the bits of the eager calls"""
    import torch
    H, W = 272, 480
    space, q, b = "YCbCr", (30, 95), (4, 128)
    rgb = torch.from_numpy(synth(H, W, seed=23)).cuda().unsqueeze(0)

    def run():
        enc = codec.encode(rgb, space, q, b, instance=2200)
        pk = codec.pack(enc, space, q, b, instance=2200)
        coef = codec.unpack(pk, 1, H, W, space, q, b, instance=2200)
        return enc, pk, coef, codec.decode(coef, enc.leaves, enc.counts, 1, H, W, space, q, b, instance=2200)

    def used(enc, pk, coef, res):                         # the parts of the buffers the calls write
        c, pc = enc.counts.cpu().numpy(), pk.counts.cpu().numpy()
        out = [enc.counts.clone(), pk.counts.clone(), res.clone()]
        for l in range(3):
            nnz, _, _, nw = (int(x) for x in pc[0, l])
            out += [pk.mask[l][0, :nw].clone(), pk.vals[l][0, :nnz].clone(), coef[l][0, :int(c[0, l, 2])].clone()]
        return out

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eager = run()
    torch.cuda.synchronize()
    eager = used(*eager)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        enc, pk, coef, res = run()
    for t in [enc.counts, pk.counts, res] + pk.mask + pk.vals + coef:
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    got = used(enc, pk, coef, res)
    assert all(torch.equal(a, e) for a, e in zip(got, eager))


def test_two_stream_roundtrip_equals_single_stream(codec):
    """DeviceCodec.roundtrip_device spreads a batch over two CUDA streams (two plans): same bits as one plan, one stream."""
    import torch
    H, W = 272, 480
    space, q, b = "YCbCr", (30, 95), (4, 128)
    batch = torch.from_numpy(np.stack([synth(H, W, seed=s) for s in range(6)])).cuda()
    one = codec.decode_encoded(codec.encode(batch, space, q, b), space, q, b).clone()
    for n in (2, 3):
        parts = codec.roundtrip_device(batch, space, q, b, streams=n)
        torch.cuda.synchronize()
        assert torch.equal(torch.cat(parts), one)
    parts8 = codec.roundtrip_device((batch * 255).to(torch.uint8), space, q, b, streams=2, out="u8")
    ref8 = codec.decode_encoded(codec.encode((batch * 255).to(torch.uint8), space, q, b), space, q, b, out="u8")
    torch.cuda.synchronize()
    assert torch.equal(torch.cat(parts8), ref8)


def test_halo_split_two_gpus_over_peer_memory():
    """SURVEY 8e on real hardware: two ranks (torchrun), each with a band of one image, halo rows / partial histograms read from
    the neighbour's workspace over NVLink, device-side barriers -- streams and decoded rows identical to the single-GPU run.
    Needs two GPUs in one box (skipped otherwise; tests/multi_gpu_halo.py is the script, bench.py --gpus N repeats it at 8192^2)."""
    import json
    import os
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                          "--master-port", "29541", os.path.join(root, "tests", "multi_gpu_halo.py"), "1024", "1280"],
                         capture_output=True, text=True, timeout=600, env=dict(os.environ, MASTER_ADDR="127.0.0.1"))
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-1500:]
    line = [l for l in out.stdout.splitlines() if l.startswith('{"halo_split"')][-1]
    res = json.loads(line)["halo_split"]
    assert all(v["identical_to_single_gpu"] for v in res["results"].values())


@pytest.mark.parametrize("space", ["OKLAB", "ICaCb", "ICtCp", "JzAzBz"])
def test_fast_transfer_functions_equal_exact_path(st, codec, space):
    """The table-driven transfer functions (csrc/powtab.h, pqfast.h) must give, bit for bit, what the exact float64 path gives:
    8-bit colours (random, the grey ramp, the dark corner of the cube where the PQ decoder clamps), then the inverse on those
    results perturbed the way quantisation perturbs them -- forward and inverse, pixel kernels and the fused 4K-style kernels."""
    import torch
    from aeaj import native
    rng = np.random.default_rng(5)
    n = 3_000_000
    rgb8 = np.concatenate([rng.integers(0, 256, (n, 3)), np.repeat(np.arange(256)[:, None], 3, 1),
                           rng.integers(0, 6, (200_000, 3)), np.zeros((1000, 3), dtype=np.int64)]).astype(np.float32) / np.float32(255.0)

    def both(x, inverse):
        out = []
        for on in (1, 0):
            native.check(st.lib.aeaj_set_fast_transfer(st.handle, on), "aeaj_set_fast_transfer")
            out.append(st.color(space, x, inverse))
        return out
    try:
        fwd_fast, fwd_exact = both(rgb8, False)
        assert np.array_equal(fwd_fast.view(np.uint32), fwd_exact.view(np.uint32)), space
        noisy = fwd_exact + (rng.standard_normal(fwd_exact.shape) * np.abs(fwd_exact).mean(0) * 0.02).astype(np.float32)
        noisy[::7] = fwd_exact[::7]
        inv_fast, inv_exact = both(noisy, True)
        assert np.array_equal(inv_fast.view(np.uint32), inv_exact.view(np.uint32)), space     # NaN -> 1.0 (T-NAN) included
        # the fused kernels (planar forward with chroma subsampling, upsampling inverse) on an image
        img = torch.from_numpy(np.stack([synth(270, 480, seed=s) for s in (1, 2)])).cuda()
        res = []
        for on in (1, 0):
            native.check(st.lib.aeaj_set_fast_transfer(codec.handle, on), "aeaj_set_fast_transfer")
            enc = codec.encode(img, space, (30, 95), (4, 64), taps=True)
            dec = codec.decode_encoded(enc, space, (30, 95), (4, 64))
            res.append(([t.clone() for t in enc.layers], [t.clone() for t in enc.coef], dec.clone()))
        for l in range(3):
            assert torch.equal(res[0][0][l], res[1][0][l]) and torch.equal(res[0][1][l], res[1][1][l])
        assert torch.equal(res[0][2].view(torch.int32), res[1][2].view(torch.int32))
    finally:                                                       # back to the library default
        native.check(st.lib.aeaj_set_fast_transfer(st.handle, 1), "aeaj_set_fast_transfer")
        native.check(st.lib.aeaj_set_fast_transfer(codec.handle, 1), "aeaj_set_fast_transfer")
