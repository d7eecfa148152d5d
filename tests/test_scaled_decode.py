"""Scaled decode (aeaj_decode_scaled, Jpeg.decompress(..., scale=k)) against a float64 reference of its definition.

For a layer h x w, scale k and m = min(k, block_min), a leaf (x, y, s) with t = s / m gives
    V = (1/m) C_t^T Y_t C_t / sc + mid,   Y_t = float32(coef * q) over the top-left t x t of the block (q: the size-s table),
at (y/m + r, x/m + c) of the ceil(h/m) x ceil(w/m) layer for the rows / columns that cover the leaf's valid extent.  Where
k > block_min, each cell of the ceil(h/k) x ceil(w/k) layer is the mean of the in-bounds cells of its (k/m) x (k/m) group.
A kernel sample must lie within gamma(t) (|C_t| |Y_t| |C_t|^T) / (m |sc|) + 2 ulp of V: the bound of the full IDCT
(test_dct_kernels, DESIGN.md section 2) at size t.  Box means: the mean of their cells' bounds, plus n u of the mean of
|V| for the float32 sum of n cells, plus the ulp of the division.

The CPU tests check the reference itself; the GPU tests compare the device's scaled layer taps with it, the colour tail
with the oracle, and scale 1 with today's decode, bit for bit.
"""
import ctypes as C

import numpy as np
import pytest

import oracle as O
from synth import synth
from test_dct_kernels import blocks_of, dct_matrix, gamma, inverse_reference, sandwich

U = 2.0 ** -24
SCALES = (2, 4, 8)
SPACES7 = ("YCbCr", "YCoCg", "YCoCg-R", "OKLAB", "ICaCb", "ICtCp", "JzAzBz")
LINEAR = ("YCbCr", "YCoCg", "YCoCg-R")


# ------------------------------------------------------------------------------------------------
# the float64 reference of the definition
# ------------------------------------------------------------------------------------------------
def natural_blocks(blocks: np.ndarray, S: int, zigzag: bool) -> np.ndarray:
    """[n, S*S] blocks in stream order -> row-major order"""
    if not zigzag:
        return blocks
    out = np.empty_like(blocks)
    out[:, O.zigzag(S).astype(np.int64)] = blocks
    return out


def scaled_layer_reference(coef, leaves, tabs, h, w, mid, sc, k, bmin, zigzag=False):
    """(V, bound) float64 planes of the 1/m layer, m = min(k, bmin); leaves [n, 4] with coefficient offsets"""
    m = min(k, bmin)
    hm, wm = -(-h // m), -(-w // m)
    V = np.full((hm, wm), np.nan)
    T = np.zeros((hm, wm))
    for S in np.unique(leaves[:, 2]):
        S = int(S)
        lv = leaves[leaves[:, 2] == S]
        t = S // m
        nat = natural_blocks(blocks_of(coef, lv, S), S, zigzag)
        Y = (nat.astype(np.int64) * tabs[S].reshape(1, -1).astype(np.int64)).astype(np.float32).astype(np.float64)
        Y = Y.reshape(-1, S, S)[:, :t, :t]
        Ct = dct_matrix(t)
        v = sandwich(Ct.T, Y, Ct) / m / float(np.float32(sc)) + float(np.float32(mid))
        e = gamma(t, False) * sandwich(np.abs(Ct).T, np.abs(Y), np.abs(Ct)) / (m * abs(float(np.float32(sc))))
        e += 2 * np.spacing(np.abs(v).astype(np.float32)).astype(np.float64)
        ar = np.arange(t)
        R = np.broadcast_to(lv[:, 1].astype(np.int64)[:, None, None] // m + ar[None, :, None], v.shape)
        Cc = np.broadcast_to(lv[:, 0].astype(np.int64)[:, None, None] // m + ar[None, None, :], v.shape)
        sel = (R < hm) & (Cc < wm)
        V[R[sel], Cc[sel]] = v[sel]
        T[R[sel], Cc[sel]] = e[sel]
    return V, T


def box_reduce_reference(plane: np.ndarray, f: int):
    """mean of the in-bounds cells of every f x f group, and the number of cells of each group"""
    h, w = plane.shape
    dh, dw = -(-h // f), -(-w // f)
    out = np.zeros((dh, dw))
    n = np.zeros((dh, dw))
    for oy in range(dh):
        for ox in range(dw):
            g = plane[oy * f:(oy + 1) * f, ox * f:(ox + 1) * f]
            out[oy, ox] = g.mean()
            n[oy, ox] = g.size
    return out, n


def scaled_reference(coef, leaves, tabs, h, w, mid, sc, k, bmin, zigzag=False):
    """(V, bound) of the final 1/k layer"""
    V, T = scaled_layer_reference(coef, leaves, tabs, h, w, mid, sc, k, bmin, zigzag)
    m = min(k, bmin)
    if k == m:
        return V, T
    Vk, n = box_reduce_reference(V, k // m)
    Tk, _ = box_reduce_reference(T, k // m)
    Ak, _ = box_reduce_reference(np.abs(V), k // m)
    return Vk, Tk + n * U * Ak + np.spacing(np.abs(Vk).astype(np.float32)).astype(np.float64)


# ------------------------------------------------------------------------------------------------
# 1. the reference itself (CPU)
# ------------------------------------------------------------------------------------------------
def _layer_case(H=203, W=331, brange=(2, 128), q=(60, 95), space="YCbCr", seed=7):
    rgb = synth(H, W, seed=seed)
    lay = O.color_forward(space, rgb.reshape(-1, 3)).reshape(H, W, 3)[..., 0]
    lay = np.ascontiguousarray(O.downsample(np.ascontiguousarray(lay), *O.layer_shapes(H, W, space)[0]))
    leaves, _, _ = O.quadtree(O.canny(lay), brange[1], brange[0])
    tabs = O.qtables(space, q, brange)[0]
    coef = O.encode_blocks(lay, space, 0, leaves, tabs)
    off = np.concatenate([[0], np.cumsum(leaves[:, 2].astype(np.int64) ** 2)])[:-1]
    lv4 = np.concatenate([leaves[:, :3], off[:, None]], axis=1).astype(np.int32)
    mid, sc = (float(v[0]) for v in O.NORM[space])
    return lay.shape, coef, lv4, tabs, mid, sc


@pytest.mark.parametrize("zigzag", [False, True])
def test_reference_scale_one_is_the_full_idct(zigzag):
    """with m = 1 the reference is inverse_reference, placed at the leaves' positions (both stream layouts)"""
    (h, w), coef, lv, tabs, mid, sc = _layer_case()
    if zigzag:
        coef = O.zigzag_stream(coef, lv)
    V, _ = scaled_layer_reference(coef, lv, tabs, h, w, mid, sc, 1, 2, zigzag)
    plain = coef if not zigzag else O.zigzag_stream(coef, lv, inverse=True)
    for S in np.unique(lv[:, 2]):
        S = int(S)
        sel = lv[lv[:, 2] == S]
        ref, _ = inverse_reference(blocks_of(plain, sel, S), tabs[S], S, mid, sc)
        for (x, y, _, _), blk in zip(sel, ref):
            bh, bw = min(S, h - y), min(S, w - x)
            assert np.array_equal(V[y:y + bh, x:x + bw], blk[:bh, :bw])


@pytest.mark.parametrize("S", (2, 4, 8, 16, 32, 64, 128, 256))
def test_reference_dc_block_gives_the_leaf_mean(S):
    """a DC-only block decodes to the constant Y00 / S (the leaf's mean) at every t = S / m"""
    q = np.ones((S, S), dtype=np.int32)
    coef = np.zeros(S * S, dtype=np.int32)
    coef[0] = 37 * S
    lv = np.array([[0, 0, S, 0]], dtype=np.int32)
    want = 37.0 / 1.5 + 0.25
    for m in (1, 2, 4, 8):
        if m > S:
            continue
        V, _ = scaled_layer_reference(coef, lv, {S: q}, S, S, 0.25, 1.5, m, m)
        assert V.shape == (S // m, S // m)
        assert np.allclose(V, want, rtol=0, atol=1e-12), (S, m)


def test_reference_box_reduce_partial_groups():
    """5 x 7 plane, groups of 2 x 2: the border groups average only the cells that exist"""
    p = np.arange(35, dtype=np.float64).reshape(5, 7) ** 1.5
    out, n = box_reduce_reference(p, 2)
    assert out.shape == (3, 4)
    assert out[0, 0] == (p[0, 0] + p[0, 1] + p[1, 0] + p[1, 1]) / 4
    assert out[0, 3] == (p[0, 6] + p[1, 6]) / 2
    assert out[2, 0] == (p[4, 0] + p[4, 1]) / 2
    assert out[2, 3] == p[4, 6]
    assert n[2, 3] == 1 and n[1, 1] == 4


def test_bad_scale_raises_before_device_work():
    from jpeg import Jpeg, JpegCompressionSettings
    with pytest.raises(ValueError):
        Jpeg(JpegCompressionSettings()).decompress(b"not even a header", scale=3)
    with pytest.raises(ValueError):
        Jpeg(JpegCompressionSettings(), deflate="device").decompress_batch([b""], scale=16)


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _need_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


@pytest.fixture(scope="module")
def codec():
    _need_cuda()
    from aeaj.codec import get_codec
    return get_codec(0)


def _encode(codec, H, W, space, q, b, zigzag, seed=5, B=1):
    import torch
    rgb = torch.from_numpy(np.stack([synth(H, W, seed=seed + i) for i in range(B)])).cuda()
    enc = codec.encode(rgb, space, q, b, stream=zigzag)
    return enc, codec.download(enc)


def _check_layers(codec, enc, host, H, W, space, q, b, k, tag):
    """the device's scaled layer taps against the reference, every layer of every image"""
    B = enc.shape[0]
    _, tl = codec.decode(enc.coef, enc.leaves, enc.counts, B, H, W, space, q, b, taps=True, zigzag=enc.zigzag, scale=k)
    codec.check_status(codec.last_decode_status, "decode")
    tabs = O.qtables(space, q, b)
    shapes = O.layer_shapes(H, W, space)
    worst = 0.0
    for i in range(B):
        for l in range(3):
            h, w = shapes[l]
            mid, sc = (float(v[l]) for v in O.NORM[space])
            L = host[i][l]
            V, T = scaled_reference(L["coef"], L["leaves"], tabs[l], h, w, mid, sc, k, b[0], enc.zigzag)
            g = tl[l][i].cpu().numpy()
            assert g.shape == (-(-h // k), -(-w // k)), tag
            assert np.isfinite(V).all(), f"{tag}: the leaves do not cover layer {l}"
            err = np.abs(g.astype(np.float64) - V)
            bad = err > T
            if bad.any():
                r, c = np.argwhere(bad)[0]
                raise AssertionError(f"{tag} layer {l}: {int(bad.sum())} samples outside the bound; first ({r}, {c}) got {g[r, c]!r} "
                                     f"want {V[r, c]!r} bound {T[r, c]!r}")
            worst = max(worst, float((err / T).max()))
    return worst


@pytest.mark.gpu
@pytest.mark.parametrize("zigzag", [False, True])
@pytest.mark.parametrize("S", (2, 4, 8, 16, 32, 64, 128, 256))
def test_every_class_every_scale(codec, S, zigzag):
    """brange (S, S) tiles the odd 333 x 517 frame with S x S leaves, partial at the borders: every size class at every scale,
    t = S / min(k, S) from 1 to 128, and the box reduce where k > S"""
    H, W, space, q = 333, 517, "YCbCr", (30, 95)
    enc, host = _encode(codec, H, W, space, q, (S, S), zigzag)
    for k in SCALES:
        r = _check_layers(codec, enc, host, H, W, space, q, (S, S), k, f"S={S} k={k} zigzag={zigzag}")
        print(f"[scaled] S={S:3d} k={k} zigzag={int(zigzag)}: max err/bound {r:.3g}")


@pytest.mark.gpu
@pytest.mark.parametrize("H,W,space,q,b", [(333, 517, "YCbCr", (30, 95), (2, 64)), (333, 517, "ICtCp", (40, 80), (4, 128)),
                                           (37, 2, "YCbCr", (30, 95), (2, 8)), (300, 260, "YCbCr", (30, 95), (2, 256))])
def test_mixed_block_ranges(codec, H, W, space, q, b):
    """mixed leaf sizes, box reduce where k > block_min (b2-64 and b4-128 at k = 8), a 37-row sliver and the b2-256 range"""
    for zigzag in (False, True):
        enc, host = _encode(codec, H, W, space, q, b, zigzag, B=2)
        for k in SCALES:
            _check_layers(codec, enc, host, H, W, space, q, b, k, f"{H}x{W} {space} b{b} k={k} zigzag={zigzag}")


@pytest.mark.gpu
def test_golden_b2_256_layers(codec, golden):
    """the reference-written synth300x260_YCbCr_b2_256 file, its leaves and coefficients, at every scale"""
    from jpeg import Jpeg, JpegCompressionSettings
    from test_device_inflate import _load_ajpg
    name = "synth300x260_YCbCr_b2_256"
    c = golden.case(name)
    j = Jpeg(JpegCompressionSettings(c["space"], tuple(c["quality"]), tuple(c["blocks"])))
    parsed = j._entropy_decode(_load_ajpg(name))
    H, W, q, b = parsed["H"], parsed["W"], parsed["quality"], parsed["blocks"]
    coef, leaves, counts = codec.upload_for_decode([parsed["layers"]], 1, H, W, c["space"], q, b)

    class Enc:
        shape, zigzag = (1, H, W), True
    enc = Enc()
    enc.coef, enc.leaves, enc.counts = coef, leaves, counts
    host = [[dict(coef=L["coef"], leaves=L["leaves"]) for L in parsed["layers"]]]
    for k in SCALES:
        _check_layers(codec, enc, host, H, W, c["space"], q, b, k, f"{name} k={k}")


@pytest.mark.gpu
@pytest.mark.parametrize("space", SPACES7)
def test_colour_tail_against_oracle(codec, space):
    """oracle.resize_linear + oracle.color_inverse of the GPU's own scaled layers: bit-exact in linear spaces, 5e-5 for PQ /
    OKLAB, <= 1 LSB in uint8, with the full decode's exclusion of the near-black NaN class in the PQ spaces.  512 x 768 at k = 2 takes the 2x chroma fast path (YCbCr, YCoCg...), k = 8 the general one."""
    H, W, q, b = 512, 768, (30, 95), (4, 64)
    enc, _ = _encode(codec, H, W, space, q, b, True, B=2)
    for k in (2, 8):
        (rgb, rgb8), tl = codec.decode(enc.coef, enc.leaves, enc.counts, 2, H, W, space, q, b, taps=True, zigzag=True, out="both", scale=k)
        codec.check_status(codec.last_decode_status, "decode")
        Hs, Ws = -(-H // k), -(-W // k)
        assert rgb.shape == (2, Hs, Ws, 3)
        for i in range(2):
            lay = [O.resize_linear(np.ascontiguousarray(tl[l][i].cpu().numpy()), Hs, Ws) for l in range(3)]
            ref = O.color_inverse(space, np.stack(lay, axis=-1).reshape(-1, 3)).reshape(Hs, Ws, 3)
            got = rgb[i].cpu().numpy()
            diff = np.abs(got.astype(np.float64) - ref.astype(np.float64))
            lsb = np.abs(rgb8[i].cpu().numpy().astype(int) - (ref * 255).astype(np.uint8).astype(int))
            if space in ("ICaCb", "ICtCp", "JzAzBz"):
                # class T-NAN of the full decode's parity test: near black, L'M'S' can land a hair below zero on one side and
                # the reference's pow then gives NaN, which its clamp turns into a white pixel; such pixels are excluded (and bounded)
                nan_class = np.all(got == 1.0, axis=-1) | np.all(ref == 1.0, axis=-1)
                assert nan_class.mean() < 2e-3, (space, k)
                diff[nan_class] = 0
                lsb[nan_class] = 0
            d = diff.max()
            assert d == 0 if space in LINEAR else d <= 5e-5, (space, k, d)
            assert lsb.max() <= 1, (space, k, lsb.max())
            assert np.array_equal(rgb8[i].cpu().numpy(), (got * 255).astype(np.uint8)), (space, k)


def _files(n=3, H=180, W=244, space="YCoCg", q=(40, 80), b=(4, 64), deflate="host"):
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    st = JpegCompressionSettings(space, q, b)
    return [Jpeg(st, deflate=deflate).compress(Image.from_array(synth(H, W, seed=40 + i), None, ".png")) for i in range(n)]


@pytest.mark.gpu
def test_scale_one_is_todays_decode(codec):
    """decompress(b, scale=1) and aeaj_decode_scaled(..., 1, ...) are bit-identical to decompress(b), f32 and u8, both inflates"""
    import torch
    from jpeg import Jpeg, JpegCompressionSettings
    blob = _files(1, deflate="device")[0]
    for deflate in ("host", "device"):
        j = Jpeg(JpegCompressionSettings(), deflate=deflate)
        a, s1 = j.decompress(blob), j.decompress(blob, scale=1)
        assert np.array_equal(a.data, s1.data) and a.original_shape == s1.original_shape
        assert np.array_equal(j.decompress_uint8(blob), j.decompress_uint8(blob, scale=1))
    H, W, space, q, b = 272, 480, "YCbCr", (30, 95), (4, 128)
    enc, _ = _encode(codec, H, W, space, q, b, True)
    full, full8 = (t.clone() for t in codec.decode_encoded(enc, space, q, b, out="both"))
    p = codec._plan(1, H, W, space, b, q)
    io = _io(enc, p.rgb_out, p.rgb8_out, p.dec_status)
    p.rgb_out.zero_(); p.rgb8_out.zero_()
    assert codec.lib.aeaj_decode_scaled(p.ptr, C.byref(io), 1, p.workspace.data_ptr(), None, torch.cuda.current_stream().cuda_stream) == 0
    assert torch.equal(p.rgb_out, full) and torch.equal(p.rgb8_out, full8)


def _io(enc, rgb, rgb8, status):
    from aeaj import native
    io = native.DecodeIO()
    for l in range(3):
        io.coef[l], io.leaves[l] = enc.coef[l].data_ptr(), enc.leaves[l].data_ptr()
    io.counts = enc.counts.data_ptr()
    io.rgb = rgb.data_ptr() if rgb is not None else None
    io.rgb_u8 = rgb8.data_ptr() if rgb8 is not None else None
    io.status = status.data_ptr()
    return io


def _leaf_means(plane, lv, s, f):
    """mean of each leaf's block of size s / f at (y / f, x / f)"""
    t = s // f
    return np.array([plane[y // f:y // f + t, x // f:x // f + t].astype(np.float64).mean() for x, y, _, _ in lv])


@pytest.mark.gpu
def test_mean_invariant_natural(codec, golden):
    """On the natural golden images, every interior leaf with s >= k keeps its mean: the mean of its scaled block equals that
    of its full-resolution block (full-decode taps).  Both are float32 evaluations of DC / (s sc) + mid; each sample errs by at
    most gamma(s) (2/s) sum|Y_s| / |sc| + 2 ulp (|C_s| <= sqrt(2/s), and the scaled path's gamma(t) (2/t) sum|Y_t| / (m |sc|)
    is smaller), so the two means differ by at most twice that, plus k^2 u max|V| for the float32 sums of the box reduce (their
    float64 averaging here adds nothing of that order).  With k > block_min, a leaf with s < k shares its cells with its
    neighbours, so the leaves checked are those with s >= k (every one with s >= m where k <= block_min)."""
    for name in golden.natural_cases:
        c = golden.case(name)
        space, q, b = c["space"], tuple(c["quality"]), tuple(c["blocks"])
        import torch
        rgb = torch.from_numpy(golden.input_f32(name)).cuda()
        H, W = rgb.shape[:2]
        enc = codec.encode(rgb, space, q, b)
        host = codec.download(enc)[0]
        _, full = codec.decode(enc.coef, enc.leaves, enc.counts, 1, H, W, space, q, b, taps=True)
        full = [t[0].cpu().numpy() for t in full]
        tabs = O.qtables(space, q, b)
        for k in SCALES:
            _, tl = codec.decode(enc.coef, enc.leaves, enc.counts, 1, H, W, space, q, b, taps=True, scale=k)
            codec.check_status(codec.last_decode_status, "decode")
            for l in range(3):
                h, w = full[l].shape
                mid, sc = (float(v[l]) for v in O.NORM[space])
                lv = host[l]["leaves"]
                for S in np.unique(lv[:, 2]):
                    S = int(S)
                    sel = lv[(lv[:, 2] == S) & (lv[:, 0] + S <= w) & (lv[:, 1] + S <= h)]
                    if S < k or not len(sel):
                        continue
                    Y = np.abs((blocks_of(host[l]["coef"], sel, S).astype(np.int64) * tabs[l][S].reshape(1, -1)).astype(np.float32))
                    vmax = max(np.abs(full[l]).max(), np.abs(tl[l][0].cpu().numpy()).max())
                    tol = 2 * (gamma(S, False) * (2.0 / S) * Y.sum(axis=1).astype(np.float64) / abs(sc)
                               + 2 * float(np.spacing(np.float32(vmax))) + k * k * U * float(vmax))
                    a = _leaf_means(full[l], sel, S, 1)
                    g = _leaf_means(tl[l][0].cpu().numpy(), sel, S, k)
                    assert (np.abs(a - g) <= tol).all(), (name, k, l, S, float(np.abs(a - g).max()))


@pytest.mark.gpu
def test_paths_agree(codec, golden):
    """host and device inflate give identical scaled images; a mixed-shape batch decodes per shape; as_uint8 is the truncation
    of the float32 output; the reference-written golden .ajpg files decode at every scale"""
    from jpeg import Jpeg, JpegCompressionSettings
    from test_device_inflate import _golden_names, _load_ajpg
    files = _files(2, deflate="device") + _files(2, 97, 131, "ICtCp", (30, 95), (2, 32)) + [_load_ajpg(n) for n in _golden_names()[:6]]
    for k in SCALES:
        jh, jd = Jpeg(JpegCompressionSettings()), Jpeg(JpegCompressionSettings(), deflate="device")
        a, d = jh.decompress_batch(files, scale=k), jd.decompress_batch(files, scale=k)
        u8 = jd.decompress_batch(files, as_uint8=True, scale=k)
        for f, x, y, z in zip(files, a, d, u8):
            full = jh.decompress(f)
            H, W = full.original_shape[:2]
            assert x.original_shape == (-(-H // k), -(-W // k), 3)
            assert x.extension == full.extension
            assert np.array_equal(x.data, y.data)
            assert np.array_equal(z, (x.data.reshape(z.shape) * 255).astype(np.uint8))
        jh.decompress(files[-1], scale=k)
        assert tuple(jh.layer_shape) == tuple(jh.decompress(files[-1]).original_shape[:2])    # the file's full size


@pytest.mark.gpu
def test_corrupt_leaves_counted(codec):
    """a leaf that does not fit the plan is skipped by the scaled path too and counted in status[3]"""
    H, W, space, q, b = 200, 328, "YCbCr", (30, 95), (4, 64)
    enc, _ = _encode(codec, H, W, space, q, b, False)
    enc.leaves[0][0, 0, 2] = 12                       # not a power of two
    enc.leaves[0][0, 1, 0] = W + 5                    # outside the layer
    codec.decode(enc.coef, enc.leaves, enc.counts, 1, H, W, space, q, b, scale=4)
    assert int(codec.last_decode_status[3].item()) == 2
    with pytest.raises(ValueError):
        codec.check_status(codec.last_decode_status, "decode")


@pytest.mark.gpu
def test_einval(codec):
    """bad scales, NULL buffers and a plan with peers are rejected with AEAJ_EINVAL"""
    import torch
    H, W, space, q, b = 128, 192, "YCbCr", (30, 95), (4, 64)
    enc, _ = _encode(codec, H, W, space, q, b, False)
    p = codec._plan(1, H, W, space, b, q, instance=3300)
    sc = codec._scaled(p, 2)
    s = torch.cuda.current_stream().cuda_stream
    lib = codec.lib
    io = _io(enc, sc.rgb_out, None, p.dec_status)
    for bad in (0, 3, 16, -2):
        assert lib.aeaj_decode_scaled(p.ptr, C.byref(io), bad, p.workspace.data_ptr(), sc.scratch.data_ptr(), s) == -1
        oh = C.c_int()
        lh = (C.c_int * 3)()
        n = C.c_int64()
        assert lib.aeaj_decode_scaled_geometry(p.ptr, bad, C.byref(oh), C.byref(oh), lh, lh, C.byref(n)) == -1
    assert lib.aeaj_decode_scaled(p.ptr, C.byref(io), 2, p.workspace.data_ptr(), None, s) == -1
    assert lib.aeaj_decode_scaled(p.ptr, C.byref(io), 2, None, sc.scratch.data_ptr(), s) == -1
    assert lib.aeaj_decode_scaled(p.ptr, None, 2, p.workspace.data_ptr(), sc.scratch.data_ptr(), s) == -1
    io_none = _io(enc, None, None, p.dec_status)
    assert lib.aeaj_decode_scaled(p.ptr, C.byref(io_none), 2, p.workspace.data_ptr(), sc.scratch.data_ptr(), s) == -1
    io.coef[1] = None
    assert lib.aeaj_decode_scaled(p.ptr, C.byref(io), 2, p.workspace.data_ptr(), sc.scratch.data_ptr(), s) == -1
    io = _io(enc, sc.rgb_out, None, p.dec_status)
    flags = torch.zeros(64, dtype=torch.int32, device="cuda")
    ws2 = (C.c_void_p * 2)(p.workspace.data_ptr(), p.workspace.data_ptr() + 256)
    fl2 = (C.c_void_p * 2)(flags.data_ptr(), flags.data_ptr() + 128)
    assert lib.aeaj_plan_set_peers(p.ptr, 0, 2, ws2, fl2) == 0
    try:
        assert lib.aeaj_decode_scaled(p.ptr, C.byref(io), 2, p.workspace.data_ptr(), sc.scratch.data_ptr(), s) == -1
    finally:
        assert lib.aeaj_plan_set_peers(p.ptr, 0, 1, None, None) == 0
    assert lib.aeaj_decode_scaled(p.ptr, C.byref(io), 2, p.workspace.data_ptr(), sc.scratch.data_ptr(), s) == 0
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_cuda_graph_capture(codec):
    """steady-state scaled decodes upload nothing, also when they alternate with full decodes: captured and replayed, they
    give the eager bits"""
    import torch
    H, W, space, q, b = 272, 480, "YCbCr", (30, 95), (4, 128)
    rgb = torch.from_numpy(synth(H, W, seed=8)).cuda().unsqueeze(0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())

    def run():
        enc = codec.encode(rgb, space, q, b, instance=4400, stream=True)
        full = codec.decode(enc.coef, enc.leaves, enc.counts, 1, H, W, space, q, b, instance=4400, zigzag=True)
        return full, [codec.decode(enc.coef, enc.leaves, enc.counts, 1, H, W, space, q, b, instance=4400, zigzag=True, out="both",
                                   scale=k) for k in SCALES]

    with torch.cuda.stream(side):
        full, outs = run()
    torch.cuda.synchronize()
    eager = [full.clone()] + [t.clone() for pair in outs for t in pair]
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        full, outs = run()
    got = [full] + [t for pair in outs for t in pair]
    for t in got:
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, e) for a, e in zip(got, eager))
