"""Every DCT / IDCT kernel against a float64 reference with an a-priori error bound.

The reference (numpy, CPU) extracts each leaf as the kernels do (np.pad 'reflect', jpeg.py:387-404), normalises it in
float32 with two rounded operations, then computes Z = C X C^T in float64.  The inverse takes Y = float32(coef * q) and
returns V = (C^T Y C) / sc + mid in float64, cropped like ao_decode_blocks.  The bound on a kernel's error is, element by
element,  E = gamma * (|C| |X| |C|^T)  (see `gamma`).  Acceptance:

  forward   |k_gpu - Z/q| <= 1/2 + E/q        a coefficient may differ from rint(Z/q) only where Z lies within E of a tie
  inverse   |g - V| <= E/|sc| + 2 ulp(V)

The CPU tests check the reference itself (against the oracle) and that the bound would catch a kernel that dropped
the 3xTF32 compensation.  The GPU tests run every size class on every kernel that serves it, the tensor-core kernels
in their steady state (at least 4 super-tiles per CTA), the partial-leaf and misaligned-store paths, the exact
quantiser on ties, and the halo-split band filter.  Run with -s to see per (class, kernel, mask): tiles per CTA, tie
flips against rint(Z/q), and the largest error seen as a fraction of its bound.
"""
import math

import numpy as np
import pytest

import oracle as O
from synth import synth

U = 2.0 ** -24
TC_CLASSES = (16, 32, 64, 128)
ALL_CLASSES = (2, 4, 8, 16, 32, 64, 128, 256)
SPACES = ("YCbCr", "YCoCg-R", "ICtCp")          # ICtCp: a PQ space, with its own mid / scale
QUALITIES = ((99, 99), (1, 1))                  # q ~ 1 everywhere / large q
STEADY_SHAPE = (1920, 2320)                     # batch 2: >= 5 super-tiles per CTA on 148 SMs for every tensor-core class
STEADY_TILES_PER_CTA = 4                        # every Out buffer and every mbarrier phase used twice


def gamma(S: int, tensor_core: bool) -> float:
    """Relative bound on a kernel's Z (or C^T Y C), as a multiple of |C| |X| |C|^T.

    FP32 kernels (k_dct_rows, k_dct_cta, k_dct256): each output is two chained dot products of length S.  With
    u = 2^-24, a float32 dot product of length n satisfies |fl(a.b) - a.b| <= n u sum|a_i b_i| (to first order), for any
    order of the additions.  The even / odd folding of the CTA and row kernels adds one rounded add or subtract in
    front of the products (one more u), and C itself is stored as float32 (|C32 - C| <= u |C|: one more u).  Pass one
    then errs by at most (S + 2) u |C| |X|, and pass two adds (S + 2) u |C| |X| |C|^T: gamma = (2S + 4) u.

    3xTF32 tensor-core kernels (k_dct_tc): an operand v is split as hi = tf32(v), lo = tf32(v - hi), which leaves
    |v - hi - lo| <= 2^-22 |v|, and hi.hi + hi.lo + lo.hi drops lo.lo, |lo_a lo_b| <= 2^-22 |a b|.  Per product that is
    at most 3 * 2^-22 relative; it happens in GEMM1 (C and X split), in GEMM2 (W and C split) and once more where W is
    split in place: < 2^-19 in all.  The accumulation in tensor memory rounds once per MMA, 3 MMAs per K step of 8, so
    3S/8 roundings per dot product; even at 2u each (truncation, which the PTX ISA does not exclude) that is below the
    (S + 2) u of the FP32 term.  Hence gamma = (2S + 4) u + 2^-19.
    """
    return (2 * S + 4) * U + (2.0 ** -19 if tensor_core else 0.0)


def on_tensor_cores(S: int, mask: int) -> bool:
    return S in TC_CLASSES and bool(mask & (1 << (int(math.log2(S)) - 4)))


def dct_matrix(S: int) -> np.ndarray:
    """C[k][i] = sqrt(2/S) cos(pi (2i + 1) k / 2S), row 0 scaled by 1/sqrt 2 (float64)"""
    k, i = np.arange(S)[:, None], np.arange(S)[None, :]
    c = np.sqrt(2.0 / S) * np.cos(np.pi * (2 * i + 1) * k / (2.0 * S))
    c[0] *= np.sqrt(0.5)
    return c


def pad_index(p, n):
    """np.pad(mode='reflect') source index of position p in an axis of length n (n == 1 replicates)"""
    n = np.asarray(n)
    period = np.maximum(2 * (n - 1), 1)
    r = p % period
    return np.where(n == 1, 0, np.where(r < n, r, period - r))


def extract(layer: np.ndarray, leaves: np.ndarray, S: int, mid, sc) -> np.ndarray:
    """float32 [n, S, S]: the normalised, reflect-padded leaves, (v - mid) * sc rounded after each operation"""
    h, w = layer.shape
    x, y = leaves[:, 0].astype(np.int64), leaves[:, 1].astype(np.int64)
    ar = np.arange(S)
    rows = y[:, None] + pad_index(ar[None, :], np.minimum(S, h - y)[:, None])
    cols = x[:, None] + pad_index(ar[None, :], np.minimum(S, w - x)[:, None])
    v = layer[rows[:, :, None], cols[:, None, :]]
    return (v - np.float32(mid)) * np.float32(sc)


def sandwich(A: np.ndarray, X: np.ndarray, B: np.ndarray) -> np.ndarray:
    """A @ X[i] @ B for every block of X [n, S, S] (float64), as two large GEMMs"""
    n, S, _ = X.shape
    t = (X.reshape(n * S, S) @ B).reshape(n, S, S)
    t = t.transpose(0, 2, 1).reshape(n * S, S) @ A.T
    return t.reshape(n, S, S).transpose(0, 2, 1)


def forward_reference(layer, leaves, S, mid, sc):
    """(Z, sum |C| |X| |C|^T), both float64 [n, S*S]"""
    X = extract(layer, leaves, S, mid, sc).astype(np.float64)
    C = dct_matrix(S)
    n = len(leaves)
    return sandwich(C, X, C.T).reshape(n, -1), sandwich(np.abs(C), np.abs(X), np.abs(C).T).reshape(n, -1)


def inverse_reference(coef_blocks, q, S, mid, sc):
    """(V, sum |C|^T |Y| |C|), float64 [n, S, S]; coef_blocks int [n, S*S], q int [S, S]"""
    Y = (coef_blocks.astype(np.int64) * q.reshape(1, -1).astype(np.int64)).astype(np.float32).astype(np.float64)
    Y = Y.reshape(-1, S, S)
    C = dct_matrix(S)
    V = sandwich(C.T, Y, C) / float(np.float32(sc)) + float(np.float32(mid))
    return V, sandwich(np.abs(C).T, np.abs(Y), np.abs(C))


def blocks_of(coef: np.ndarray, leaves: np.ndarray, S: int) -> np.ndarray:
    return coef[leaves[:, 3].astype(np.int64)[:, None] + np.arange(S * S)[None, :]]


def with_offsets(leaves3: np.ndarray) -> np.ndarray:
    off = np.concatenate([[0], np.cumsum(leaves3[:, 2].astype(np.int64) ** 2)])[:-1]
    return np.concatenate([leaves3[:, :3], off[:, None]], axis=1).astype(np.int32)


class Tally:
    """per (class, kernel, mask): coefficients / samples checked, tie flips, largest error / bound"""

    def __init__(self):
        self.rows = {}

    def add(self, key, n, ties, ratio):
        r = self.rows.setdefault(key, [0, 0, 0.0])
        r[0] += n
        r[1] += ties
        r[2] = max(r[2], ratio)

    def report(self, title, tiles=None):
        for key in sorted(self.rows):
            n, ties, ratio = self.rows[key]
            tl = f" tiles/CTA >= {tiles[key[0]]}" if tiles and key[0] in tiles and key[1] == "tc" else ""
            print(f"[{title}] S={key[0]:3d} {key[1]:4s} mask={key[2]:#x}: {n} checked, {ties} tie flips, "
                  f"max err/bound {ratio:.3g}{tl}")


def check_forward(got, Z, Eabs, q, g, tag):
    """got int [n, S*S], Z / Eabs float64 [n, S*S], q int [S, S].  Returns (tie flips, largest error / bound)."""
    qf = q.reshape(1, -1).astype(np.float64)
    zq = Z / qf
    E = g * Eabs
    dev = np.abs(got - zq)
    bad = dev > 0.5 + E / qf
    if bad.any():
        i, j = np.argwhere(bad)[0]
        raise AssertionError(f"{tag}: {int(bad.sum())} coefficients outside the bound; first: block {i} index {j} "
                             f"got {int(got[i, j])} Z/q {zq[i, j]!r} bound {E[i, j] / qf[0, j]!r}")
    ties = int((got != np.rint(zq)).sum())
    excess = np.clip(dev - 0.5, 0, None) * qf
    ratio = float(np.max(excess[E > 0] / E[E > 0])) if (E > 0).any() else 0.0
    return ties, ratio


def check_inverse(g_layer, V_layer, T_layer, tag):
    """g (kernel), V (reference), T (bound) over the whole layer; returns the largest error / bound"""
    assert np.isfinite(V_layer).all(), f"{tag}: the leaves do not cover the layer"
    err = np.abs(g_layer.astype(np.float64) - V_layer)
    bad = err > T_layer
    if bad.any():
        r, c = np.argwhere(bad)[0]
        raise AssertionError(f"{tag}: {int(bad.sum())} samples outside the bound; first ({r}, {c}) got {g_layer[r, c]!r} "
                             f"want {V_layer[r, c]!r} bound {T_layer[r, c]!r}")
    return float((err / T_layer).max())


def inverse_layers(blocks_by_size, leaves, tabs, mid, sc, h, w, mask):
    """reference layer V and bound layer T for the coefficient blocks {S: int [n_S, S*S]} of `leaves` (x, y, size)"""
    V_layer = np.full((h, w), np.nan)
    T_layer = np.zeros((h, w))
    for S, blocks in blocks_by_size.items():
        lv = leaves[leaves[:, 2] == S]
        V, Eabs = inverse_reference(blocks, tabs[S], S, mid, sc)
        T = gamma(S, on_tensor_cores(S, mask)) * Eabs / abs(float(np.float32(sc))) + 2 * np.spacing(np.abs(V).astype(np.float32)).astype(np.float64)
        ar = np.arange(S)
        R = np.broadcast_to(lv[:, 1].astype(np.int64)[:, None, None] + ar[None, :, None], V.shape)
        Cc = np.broadcast_to(lv[:, 0].astype(np.int64)[:, None, None] + ar[None, None, :], V.shape)
        m = (R < h) & (Cc < w)
        V_layer[R[m], Cc[m]] = V[m]
        T_layer[R[m], Cc[m]] = T[m]
    return V_layer, T_layer


def tf32(a: np.ndarray) -> np.ndarray:
    """round float32 to the nearest TF32 value (10 explicit mantissa bits), as the kernels' tf32_rn"""
    b = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xffffe000)).view(np.float32)


def _layer_and_leaves(H=200, W=328, brange=(2, 128), seed=4, space="YCbCr", channel=0):
    rgb = synth(H, W, seed=seed)
    lay = O.color_forward(space, rgb.reshape(-1, 3)).reshape(H, W, 3)[..., channel]
    lay = np.ascontiguousarray(O.downsample(np.ascontiguousarray(lay), *O.layer_shapes(H, W, space)[channel]))
    leaves, _, _ = O.quadtree(O.canny(lay), brange[1], brange[0])
    return lay, leaves


# ------------------------------------------------------------------------------------------------
# 1. the reference itself (CPU)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("space,channel", [("YCbCr", 0), ("YCoCg-R", 1), ("ICtCp", 2)])
def test_reference_matches_oracle(space, channel):
    """Z agrees with the oracle's float64 DCT rounded to float32, and V with ao_decode_blocks, within the rounding
    that the oracle applies on the way; every leaf size 2 .. 128 and partial leaves at the borders."""
    lay, leaves = _layer_and_leaves(203, 331, (2, 128), seed=7, space=space, channel=channel)
    sizes = set(leaves[:, 2].tolist())
    assert {2, 4, 8, 16}.issubset(sizes), sizes
    q = (60, 95)
    tabs = O.qtables(space, q, (2, 128))[channel]
    mid, sc = (float(v[channel]) for v in O.NORM[space])
    coef, dct = O.encode_blocks(lay, space, channel, leaves, tabs, want_dct=True)
    lv4 = with_offsets(leaves)
    h, w = lay.shape
    blocks = {}
    for S in sorted(sizes):
        sel = leaves[:, 2] == S
        Z, Eabs = forward_reference(lay, lv4[sel], S, mid, sc)
        oz = blocks_of(dct, lv4[sel], S).astype(np.float64)
        # the oracle rounds its float64 Z to float32; its own float64 sums differ from ours by far less than 2^-40
        tol = 0.5 * np.spacing(np.abs(Z).astype(np.float32)).astype(np.float64) + 2.0 ** -40 * Eabs
        assert (np.abs(oz - Z) <= tol).all(), S
        blocks[S] = blocks_of(coef, lv4[sel], S)
    V, T = inverse_layers(blocks, leaves, tabs, mid, sc, h, w, mask=0)
    ref = O.decode_blocks(coef, leaves, tabs, h, w, space, channel)
    # the oracle rounds C^T Y C to float32, then divides and adds in float32: 1/2 ulp of the sum before the division,
    # half an ulp for each of the two operations; T (gamma = 2S + 4 ulp) is far larger than the first term
    assert (np.abs(ref.astype(np.float64) - V) <= T).all()


@pytest.mark.parametrize("S", TC_CLASSES)
def test_bound_catches_uncompensated_tf32(S):
    """A single TF32 GEMM pair (operands rounded to TF32, float32 accumulation) violates the 3xTF32 bound on a clear
    fraction of the coefficients of realistic blocks: the test would notice a dropped compensation term."""
    lay, _ = _layer_and_leaves(512, 512, (4, 128), seed=9)
    leaves = np.array([(x, y, S, 0) for y in range(0, 512, S) for x in range(0, 512, S)], dtype=np.int32)
    mid, sc = (float(v[0]) for v in O.NORM["YCbCr"])
    X = extract(lay, leaves, S, mid, sc)
    Z, Eabs = forward_reference(lay, leaves, S, mid, sc)
    C32 = dct_matrix(S).astype(np.float32)
    # GEMM1 W = C X and GEMM2 Out = W C^T on TF32 operands; the products are exact in float64, the sums rounded to float32
    Wm = np.matmul(tf32(C32).astype(np.float64), tf32(X).astype(np.float64)).astype(np.float32)
    out = np.matmul(tf32(Wm).astype(np.float64), tf32(C32).T.astype(np.float64)).astype(np.float32)
    err = np.abs(out.reshape(len(leaves), -1).astype(np.float64) - Z)
    ratio = err / (gamma(S, True) * Eabs)
    frac, blocks, worst = float((ratio > 1).mean()), float((ratio > 1).any(axis=1).mean()), float(ratio.max())
    print(f"[teeth] S={S}: single TF32 violates the 3xTF32 bound on {frac:.2%} of the coefficients, in {blocks:.0%} of the "
          f"blocks, by up to {worst:.1f}x")
    # the bound grows with S (2S + 4 roundings) and the TF32 error only like sqrt(S): ~70 % of the coefficients at S = 16,
    # ~0.6 % at S = 128 -- but in every block, and any single violation fails the GPU tests
    assert blocks == 1.0 and frac > 0.0025 and worst > 4, (frac, blocks, worst)
    # ... while float32 operands with the same sums stay inside the FP32 bound
    exact = np.matmul(np.matmul(C32.astype(np.float64), X.astype(np.float64)).astype(np.float32).astype(np.float64),
                      C32.T.astype(np.float64)).astype(np.float32)
    assert (np.abs(exact.reshape(len(leaves), -1) - Z) <= gamma(S, False) * Eabs).all()


def _class_counts(H, W, space, S, B=2):
    return B * sum(math.ceil(h / S) * math.ceil(w / S) for h, w in O.layer_shapes(H, W, space))


def test_steady_state_workload_geometry():
    """The frame of the class tests gives every tensor-core CTA >= 4 super-tiles on a 148-SM B200, and some class
    ends in a partial super-tile (the GPU test asserts the same from the device's SM count and the real leaf lists)."""
    for space in SPACES:
        partial = False
        for S in TC_CLASSES:
            n = _class_counts(*STEADY_SHAPE, space, S)
            NL = (128 // S) ** 2
            assert math.ceil(n / NL) // 148 >= STEADY_TILES_PER_CTA, (space, S, n)
            partial |= n % NL != 0
        assert partial, space


# ------------------------------------------------------------------------------------------------
# GPU fixtures
# ------------------------------------------------------------------------------------------------
def _need_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")


@pytest.fixture(scope="module")
def codec():
    _need_cuda()
    from aeaj.codec import get_codec
    c = get_codec(0)
    saved = c.tensor_dct
    yield c
    c.tensor_dct = saved


@pytest.fixture
def tc(codec):
    """the codec, with its tensor-core mask restored after the test"""
    saved = codec.tensor_dct
    yield codec
    codec.tensor_dct = saved


@pytest.fixture(scope="module")
def st():
    _need_cuda()
    from aeaj.codec import get_stages
    return get_stages(0)


def _encode(codec, rgb, space, q, b, mask, **kw):
    codec.tensor_dct = mask
    enc = codec.encode(rgb, space, q, b, **kw)
    got = codec.download(enc)                    # synchronises, check_status: hysteresis, tensor-core timeout flag
    assert not codec.tensor_dct_timed_out()
    return enc, got


def _decode_taps(codec, per_image, B, H, W, space, q, b, mask, zigzag=False):
    codec.tensor_dct = mask
    up = codec.upload_for_decode(per_image, B, H, W, space, q, b)
    _, tl = codec.decode(*up, B, H, W, space, q, b, taps=True, zigzag=zigzag)
    codec.check_status(codec.last_decode_status, "decode")
    assert not codec.tensor_dct_timed_out()
    return [t.cpu().numpy() for t in tl]


def _masks(S):
    return [0] + ([1 << (int(math.log2(S)) - 4), 0xf] if S in TC_CLASSES else [])


def _kernel(S, mask):
    return "tc" if on_tensor_cores(S, mask) else "fp32"


# ------------------------------------------------------------------------------------------------
# 2 + 3. every size class on every kernel, forward and inverse, tensor cores in steady state
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("S", ALL_CLASSES)
@pytest.mark.parametrize("space", SPACES)
def test_every_class_every_kernel(tc, space, S):
    """brange = (S, S) tiles every layer with S x S leaves.  Forward: every coefficient within the bound, for mask 0
    (FP32 kernels) and the class's tensor-core bit; mask 0xf gives the same coefficients as the class bit; the .ajpg
    layout is the zigzag of the row-major result.  Inverse: the reference's own coefficients, dense random integers
    and one moving non-zero per leaf, each within the bound; the zigzag layout decodes bit-identically."""
    import torch
    codec = tc
    H, W = STEADY_SHAPE if S in TC_CLASSES else ((540, 1000) if S == 256 else (270, 484))
    B, b = 2, (S, S)
    rgb = torch.from_numpy(np.stack([synth(H, W, seed=s) for s in (31, 32)])).cuda()
    shapes = O.layer_shapes(H, W, space)
    mids, scs = O.NORM[space]
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    masks = _masks(S)
    tiles = {}
    fwd, inv = Tally(), Tally()
    ref = None                                                   # per plane: (leaves, Z, Eabs); the layer does not depend on q
    for q in QUALITIES:
        tabs = O.qtables(space, q, b)
        row = {}
        for mask in masks:
            enc, got = _encode(codec, rgb, space, q, b, mask, taps=True)
            lays = [enc.layers[l].cpu().numpy() for l in range(3)]
            if ref is None:
                ref = {}
                n = 0
                for k in range(B):
                    for l in range(3):
                        lv = got[k][l]["leaves"]
                        assert (lv[:, 2] == S).all() and np.array_equal(lv[:, 3], np.arange(len(lv)) * S * S)
                        assert lays[l][k].shape == shapes[l]
                        n += len(lv)
                        ref[k, l] = (lay0 := lays[l][k].copy(), lv) + forward_reference(lay0, lv, S, mids[l], scs[l])
                assert n == _class_counts(H, W, space, S, B)
                if S in TC_CLASSES:
                    NL = (128 // S) ** 2
                    tiles[S] = math.ceil(n / NL) // sm
                    assert tiles[S] >= STEADY_TILES_PER_CTA, (S, n, sm)
            for k in range(B):
                for l in range(3):
                    lay0, lv, Z, Eabs = ref[k, l]
                    assert np.array_equal(lays[l][k], lay0), "the colour stage output changed"
                    assert len(got[k][l]["coef"]) == len(lv) * S * S
                    blocks = got[k][l]["coef"].reshape(len(lv), S * S)
                    if mask == 0xf:                                   # the same kernel as the class bit
                        assert np.array_equal(got[k][l]["coef"], row[masks[1]][k][l]["coef"]), (space, q, k, l)
                    else:
                        ties, ratio = check_forward(blocks, Z, Eabs, tabs[l][S], gamma(S, on_tensor_cores(S, mask)),
                                                    f"{space} q={q} S={S} mask={mask:#x} image {k} layer {l}")
                        fwd.add((S, _kernel(S, mask), mask), blocks.size, ties, ratio)
            row[mask] = got
            _, gz = _encode(codec, rgb, space, q, b, mask, stream=True)
            for k in range(B):
                for l in range(3):
                    assert np.array_equal(gz[k][l]["coef"], O.zigzag_stream(got[k][l]["coef"], got[k][l]["leaves"][:, :3])), \
                        (space, q, mask, k, l)
        # ---- inverse: three inputs, every mask, both layouts
        rng = np.random.default_rng(S * 7 + len(space))
        for kind in ("own", "dense", "sparse"):
            per_image = []
            for k in range(B):
                layers = []
                for l in range(3):
                    _, lv, Z, _ = ref[k, l]
                    qt = tabs[l][S].reshape(1, -1).astype(np.int64)
                    if kind == "own":
                        cb = np.rint(Z / qt)
                    elif kind == "dense":
                        lim = (1 << 15) // qt
                        cb = rng.integers(-lim, lim + 1, size=Z.shape)
                    else:
                        cb = np.zeros(Z.shape, dtype=np.int64)
                        pos = (np.arange(len(lv)) * 37 + 11 * k + 5 * l) % (S * S)
                        lim = (1 << 15) // qt[0, pos]
                        cb[np.arange(len(lv)), pos] = rng.integers(1, lim + 1) * rng.choice([-1, 1], size=len(lv))
                    cb = cb.astype(np.int32)
                    layers.append(dict(leaves=lv, coef=cb.ravel()))
                per_image.append(layers)
            res = {}
            for mask in masks:
                res[mask] = _decode_taps(codec, per_image, B, H, W, space, q, b, mask)
            zz = [[dict(leaves=d["leaves"], coef=O.zigzag_stream(d["coef"], d["leaves"][:, :3])) for d in layers] for layers in per_image]
            for mask in masks:
                g = _decode_taps(codec, zz, B, H, W, space, q, b, mask, zigzag=True)
                for l in range(3):
                    assert np.array_equal(g[l].view(np.uint32), res[mask][l].view(np.uint32)), (kind, mask, l, "zigzag layout")
            for mask in masks:
                for k in range(B):
                    for l in range(3):
                        g = res[mask][l][k]
                        if mask == 0xf:
                            assert np.array_equal(g.view(np.uint32), res[masks[1]][l][k].view(np.uint32))
                            continue
                        lay0, lv, _, _ = ref[k, l]
                        V, T = inverse_layers({S: per_image[k][l]["coef"].reshape(len(lv), -1)}, lv, tabs[l], mids[l], scs[l],
                                              *shapes[l], mask=mask)
                        ratio = check_inverse(g, V, T, f"{space} q={q} S={S} mask={mask:#x} {kind} image {k} layer {l}")
                        inv.add((S, _kernel(S, mask), mask), g.size, 0, ratio)
    fwd.report(f"forward {space}", tiles)
    inv.report(f"inverse {space}", tiles)


# ------------------------------------------------------------------------------------------------
# 4. partial leaves, reflection folds, unaligned stores
# ------------------------------------------------------------------------------------------------
GEOM_SHAPES = [(3, 100), (100, 3), (2, 131), (131, 2), (6, 45), (7, 203), (37, 203), (200, 333)]


@pytest.mark.gpu
def test_partial_leaf_and_alignment_geometry(tc):
    """Small shapes, every class, mask 0 and 0xf, forward and inverse, against the bound.  Asserts that the cases the
    tensor-core loads and stores treat specially were reached: layers 1, 2 and 3 samples high or wide, leaves at least
    8 times taller or wider than the layer (the reflection folds many times), leaf widths that are not a multiple of 8
    (scalar IDCT store), and tensor-core leaves that follow 2 x 2 leaves in the stream."""
    import torch
    from aeaj import native
    codec = tc
    space, q = "YCbCr", (90, 99)
    mids, scs = O.NORM[space]
    branges = [(S, S) for S in ALL_CLASSES] + [(2, S) for S in TC_CLASSES]
    thin, fold, narrow, after2, unaligned = set(), set(), set(), set(), 0
    fwd, inv_worst = Tally(), {0: 0.0, 0xf: 0.0}
    cases = 0
    for H, W in GEOM_SHAPES:
        rgb = torch.from_numpy(synth(H, W, seed=H * 1000 + W)[None]).cuda()
        shapes = O.layer_shapes(H, W, space)
        for b in branges:
            if any(O.root_size(h, w) < b[0] for h, w in shapes):
                continue                                           # the plan rejects it: a layer smaller than the block size
            tabs = O.qtables(space, q, b)
            for mask in (0, 0xf):
                try:
                    enc, got = _encode(codec, rgb, space, q, b, mask, taps=True)
                except native.AeajError as e:
                    pytest.fail(f"{(H, W)} {b}: {e}")
                cases += 1
                lays = [enc.layers[l][0].cpu().numpy() for l in range(3)]
                own = []
                for l in range(3):
                    h, w = shapes[l]
                    if min(h, w) <= 3:
                        thin.add(min(h, w))
                    lv = got[0][l]["leaves"]
                    coef = got[0][l]["coef"]
                    blocks = {}
                    for S in sorted(set(lv[:, 2].tolist())):
                        sel = lv[lv[:, 2] == S]
                        Z, Eabs = forward_reference(lays[l], sel, S, mids[l], scs[l])
                        ties, ratio = check_forward(blocks_of(coef, sel, S), Z, Eabs, tabs[l][S], gamma(S, on_tensor_cores(S, mask)),
                                                    f"{(H, W)} {b} mask={mask:#x} layer {l} S={S}")
                        fwd.add((S, _kernel(S, mask), mask), Z.size, ties, ratio)
                        blocks[S] = np.rint(Z / tabs[l][S].reshape(1, -1)).astype(np.int32)
                        if on_tensor_cores(S, mask):
                            bh, bw = np.minimum(S, h - sel[:, 1]), np.minimum(S, w - sel[:, 0])
                            if (S >= 8 * np.minimum(bh, bw)).any():
                                fold.add(S)
                            if (bw % 8 != 0).any():
                                narrow.add(S)
                            if (lv[:, 2] == 2).any() and (np.nonzero(lv[:, 2] == S)[0] > np.argmax(lv[:, 2] == 2)).any():
                                after2.add(S)
                            unaligned += int((sel[:, 3] % 8 != 0).sum())
                    own.append(blocks)
                # inverse of the reference's own coefficients, in the leaf order of the stream
                ups = []
                for l in range(3):
                    lv = got[0][l]["leaves"]
                    cf = np.empty(int((lv[:, 2].astype(np.int64) ** 2).sum()), dtype=np.int32)
                    for S, bl in own[l].items():
                        sel = lv[lv[:, 2] == S]
                        cf[sel[:, 3].astype(np.int64)[:, None] + np.arange(S * S)[None, :]] = bl
                    ups.append(dict(leaves=lv, coef=cf))
                g = _decode_taps(codec, [ups], 1, H, W, space, q, b, mask)
                for l in range(3):
                    lv = got[0][l]["leaves"]
                    V, T = inverse_layers(own[l], lv, tabs[l], mids[l], scs[l], *shapes[l], mask=mask)
                    ratio = check_inverse(g[l][0], V, T, f"{(H, W)} {b} mask={mask:#x} layer {l} inverse")
                    inv_worst[mask] = max(inv_worst[mask], ratio)
    fwd.report("geometry forward")
    print(f"[geometry] {cases} cases; thin layers {sorted(thin)}, folds {sorted(fold)}, widths % 8 != 0 {sorted(narrow)}, "
          f"after 2 x 2 leaves {sorted(after2)}, offsets % 8 != 0: {unaligned}; inverse max err/bound: mask 0 "
          f"{inv_worst[0]:.3g}, mask 0xf {inv_worst[0xf]:.3g}")
    assert {1, 2, 3} <= thin
    assert set(TC_CLASSES) <= fold and set(TC_CLASSES) <= narrow and set(TC_CLASSES) <= after2
    # 2 x 2 leaves come as 2 or 4 siblings (8 or 16 coefficients); a node with a single in-bounds child holds the layer's
    # bottom-right corner, and that leaf is the last one in DFS order.  So a leaf of 16 or more starts at a multiple of 8
    # coefficients, and plane bases are multiples of top^2: the 32-byte store of the tensor-core epilogue always applies
    assert unaligned == 0


# ------------------------------------------------------------------------------------------------
# 5. the exact quantiser on ties (FP32 kernels through the stage API)
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("S", [4, 16, 64, 256])
def test_quantiser_ties_exact(st, S):
    """Constant S x S blocks with mid = 0, sc = 1: the DC weight 1/sqrt(S) is a power of two, so with at most
    24 - log2 S significant bits in the sample the FP32 kernels produce DC = S * c exactly.  DC sits on every tie
    +-(k + 1/2) q (and one step either side on the grid of such values), for q = 1 .. 255 and a few larger steps, k up to
    |DC| ~ 2^15: the quantised DC must be rint(DC / q), ties to even, exactly.  The AC coefficients follow the bound."""
    bits = 24 - int(math.log2(S))
    step = 2.0 ** (15 - bits)                       # |DC| < 2^15 on this grid has at most `bits` significant bits
    rng = np.random.default_rng(S)
    qtab = rng.integers(1, 256, size=(S, S)).astype(np.int32)
    C = dct_matrix(S)
    v, va = C.sum(axis=1), np.abs(C).sum(axis=1)    # C . 1 and |C| . 1: Z = c v v^T, |C| |X| |C|^T = |c| va va^T
    nk = 6 if S == 256 else 24
    flips_checked = 0
    worst = 0.0
    for qv in list(range(1, 256)) + [256, 257, 1000, 4095, 12345, 32767]:
        qtab[0, 0] = qv
        kmax = int((2.0 ** 15 - step) / qv - 0.5)
        ks = np.unique(np.round(np.linspace(0, max(kmax, 0), nk)).astype(np.int64))
        ties = (ks + 0.5) * qv
        dc = np.concatenate([t + d for t in (ties, -ties) for d in (-step, 0.0, step)])
        dc = dc[np.abs(dc) < 2.0 ** 15]
        c = (dc / S).astype(np.float32)
        assert np.array_equal(c.astype(np.float64) * S, dc)
        n = len(c)
        layer = np.ascontiguousarray(np.repeat(np.repeat(c[None, :], S, axis=0), S, axis=1))
        leaves = np.array([(i * S, 0, S, i * S * S) for i in range(n)], dtype=np.int32)
        got = st.dct_quant(layer, leaves, {S: qtab}, 0.0, 1.0, (S, S)).reshape(n, S * S)
        want_dc = np.rint(dc / qv).astype(np.int64)
        bad = got[:, 0] != want_dc
        assert not bad.any(), (S, qv, dc[bad][:4], got[bad, 0][:4], want_dc[bad][:4])
        flips_checked += n
        Z = c.astype(np.float64)[:, None] * np.outer(v, v).ravel()[None, :]
        Eabs = np.abs(c.astype(np.float64))[:, None] * np.outer(va, va).ravel()[None, :]
        _, ratio = check_forward(got, Z, Eabs, qtab, gamma(S, False), f"S={S} q={qv} AC")
        worst = max(worst, ratio)
    print(f"[ties] S={S}: {flips_checked} DC values on and next to ties exact; AC max err/bound {worst:.3g}")


# ------------------------------------------------------------------------------------------------
# 6. halo split with tensor cores, empty classes
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("b", [(16, 16), (32, 32), (64, 64), (128, 128), (4, 128)])
def test_halo_split_tensor_core_band_filter(tc, b):
    """TiledCodec(emulate=4) with every class on the tensor cores runs each class's kernel once per band, which keeps
    only the leaves of that band: the result equals the single call with the same mask."""
    import torch
    from aeaj.tiled import TiledCodec
    codec = tc
    H, W, space, q = 1024, 640, "YCbCr", (30, 95)
    rgb = torch.from_numpy(synth(H, W, seed=23)).cuda()
    codec.tensor_dct = 0xf
    ref = codec.download(codec.encode(rgb, space, q, b))[0]
    ref_dec = codec.decode_encoded(codec._plan(1, H, W, space, b, q).out, space, q, b)[0].clone()
    t = TiledCodec(codec, emulate=4)
    enc = t.encode(rgb, H, W, space, q, b)
    got = codec.download(enc)[0]
    assert not codec.tensor_dct_timed_out()
    for l in range(3):
        for k in ("states", "leaves", "coef"):
            assert np.array_equal(got[l][k], ref[l][k]), (b, l, k)
    assert torch.equal(t.decode(enc, H, W, space, q, b), ref_dec)
    assert not codec.tensor_dct_timed_out()


@pytest.mark.gpu
def test_empty_tensor_core_classes(tc):
    """A flat image with b16-128 has only 128 x 128 leaves: the kernels of classes 16 / 32 / 64 launch with count = 0.
    No timeout; mask 0xf gives the coefficients of mask 0 wherever no tie is within the bound, and both directions of
    both masks stay within the bound."""
    import torch
    codec = tc
    H, W, space, q, b = 600, 1000, "YCbCr", (30, 95), (16, 128)
    rgb = torch.from_numpy(np.broadcast_to(np.array([0.8, 0.35, 0.55], dtype=np.float32), (1, H, W, 3)).copy()).cuda()
    shapes = O.layer_shapes(H, W, space)
    tabs = O.qtables(space, q, b)
    mids, scs = O.NORM[space]
    res = {}
    for mask in (0, 0xf):
        enc, got = _encode(codec, rgb, space, q, b, mask, taps=True)
        res[mask] = [got[0][l]["coef"] for l in range(3)]
        ups = []
        for l in range(3):
            lv = got[0][l]["leaves"]
            assert (lv[:, 2] == 128).all()
            lay = enc.layers[l][0].cpu().numpy()
            Z, Eabs = forward_reference(lay, lv, 128, mids[l], scs[l])
            qf = tabs[l][128].reshape(1, -1)
            check_forward(blocks_of(got[0][l]["coef"], lv, 128), Z, Eabs, tabs[l][128], gamma(128, on_tensor_cores(128, mask)), f"flat mask={mask:#x}")
            if mask == 0xf:
                safe = (np.abs(Z / qf - np.rint(Z / qf)) < 0.5 - gamma(128, True) * Eabs / qf).ravel()
                assert np.array_equal(res[0xf][l][safe], res[0][l][safe])
            ups.append(dict(leaves=lv, coef=np.rint(Z / qf).astype(np.int32).ravel()))
        g = _decode_taps(codec, [ups], 1, H, W, space, q, b, mask)
        for l in range(3):
            V, T = inverse_layers({128: ups[l]["coef"].reshape(-1, 128 * 128)}, ups[l]["leaves"], tabs[l], mids[l], scs[l], *shapes[l], mask=mask)
            check_inverse(g[l][0], V, T, f"flat inverse mask={mask:#x} layer {l}")


@pytest.mark.gpu
def test_halo_split_ignores_layout_left_on_the_plan(tc):
    """The halo path shares its plan with DeviceCodec.encode for B = 1.  After encode(stream=True) on that plan it must
    still write row-major blocks, with the codec's tensor-core mask."""
    import torch
    from aeaj.tiled import TiledCodec
    codec = tc
    H, W, space, q, b = 512, 640, "YCbCr", (30, 95), (4, 128)
    rgb = torch.from_numpy(synth(H, W, seed=29)).cuda()
    ref = codec.download(codec.encode(rgb, space, q, b))[0]
    codec.download(codec.encode(rgb, space, q, b, stream=True))
    t = TiledCodec(codec, emulate=2)
    enc = t.encode(rgb, H, W, space, q, b)
    assert not enc.zigzag
    got = codec.download(enc)[0]
    for l in range(3):
        assert np.array_equal(got[l]["coef"], ref[l]["coef"]), l
