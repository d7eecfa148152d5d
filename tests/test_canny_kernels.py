"""Canny kernels (csrc/canny.cu) against OpenCV with IPP off -- the library the reference calls, DESIGN §2's mode S -- and
against a float64 bilateral, at the sizes the product runs, at CLAHE padding and kernel tile seams, across the prefilter's
packed / general regime boundary, under hysteresis stress patterns and in mixed fused batches.

References: CLAHE, Gaussian, thresholds and Canny are bit-exact against cv2 / numpy.  The bilateral is bit-exact against
the oracle's scalar model (O.bilateral5; OpenCV's vectorised bilateral differs from it on near-half ties, class T-BIL) and
equals rint of the float64 weighted mean everywhere outside a tie band of 1e-4 (3x the worst case measured for OpenCV and the
oracle), where it may be either neighbour.  The CPU self-checks pin the references against the oracle first."""
import math

import numpy as np
import pytest

import oracle as O
from synth import synth

TIE_BAND = 1e-4
HY_TW, HY_TH = 256, 32          # hysteresis tile: 8 bitmap words x 32 rows
PF_TW, PF_TH = 128, 64          # prefilter tile (halo 3)


@pytest.fixture(scope="module")
def cv():
    cv2 = pytest.importorskip("cv2")
    prev = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    yield cv2
    cv2.ipp.setUseIPP(prev)


# ------------------------------------------------------------------------------------------------
# references
# ------------------------------------------------------------------------------------------------
def ref_clahe(x):
    import cv2
    return cv2.createCLAHE(clipLimit=0.75, tileGridSize=(4, 4)).apply(x)


def ref_gauss(x):
    import cv2
    return cv2.GaussianBlur(x, (3, 3), 0)


def _reflect101(i, n):
    if n == 1:
        return 0
    while i < 0 or i >= n:
        i = -i if i < 0 else 2 * (n - 1) - i
    return i


_BIL_W64 = np.exp(-np.arange(255 * 255 + 5, dtype=np.float64) / (2 * 75.0 ** 2))   # exp(-(dv^2 + r^2) / (2 75^2)), dv^2 + r^2 integer


def ref_bilateral64(g):
    """cv.bilateralFilter(g, 5, 75, 75) in float64 before rounding: the 13 taps with r^2 <= 4, REFLECT_101 border."""
    h, w = g.shape
    ry = np.array([_reflect101(i, h) for i in range(-2, h + 2)])
    rx = np.array([_reflect101(i, w) for i in range(-2, w + 2)])
    p = g.astype(np.int32)[ry][:, rx]
    c = p[2:2 + h, 2:2 + w]
    num = np.zeros((h, w))
    den = np.zeros((h, w))
    for dy in range(-2, 3):
        for dx in range(-2, 3):
            if dy * dy + dx * dx > 4:
                continue
            v = p[2 + dy:2 + dy + h, 2 + dx:2 + dx + w]
            wt = _BIL_W64[(v - c) ** 2 + dy * dy + dx * dx]
            num += wt * v
            den += wt
    return num / den


def ref_thresholds(b):
    lo, hi = np.percentile(b, [10, 30])
    return float(lo), float(hi)


def ref_canny(b, lo, hi):
    import cv2
    return cv2.Canny(b, lo, hi, L2gradient=True, apertureSize=3) > 0


def ref_chain(layer):
    """EdgeDetection.canny: cast, CLAHE, Gaussian, bilateral (scalar model), percentile thresholds, Canny."""
    b = O.bilateral5(ref_gauss(ref_clahe(O.cast_u8(layer))))
    return ref_canny(b, *ref_thresholds(b))


def check_tie_band(got, q):
    """got == rint(q) outside the tie band; inside it floor(q) or ceil(q).  Returns the number of pixels in the band."""
    near = np.abs(q - np.floor(q) - 0.5) < TIE_BAND
    off = (got != np.rint(q)) & ~near
    assert not off.any(), f"{int(off.sum())} px off rint(q64) outside the tie band, e.g. {np.argwhere(off)[:3].tolist()}"
    qn, gn = q[near], got[near]
    assert np.all((gn == np.floor(qn)) | (gn == np.ceil(qn))), "a tie-band pixel is neither floor nor ceil of q64"
    return int(near.sum())


def first_diff(a, b):
    d = np.argwhere(np.asarray(a) != np.asarray(b))
    return f"{len(d)} px differ, first at {d[:3].tolist()}"


# ------------------------------------------------------------------------------------------------
# the prefilter's regime predicate, restated: clahe_geom and two_ok / uniform of k_prefilter
# ------------------------------------------------------------------------------------------------
def clahe_geom(h, w):
    eh, ew = h, w
    if w % 4 or h % 4:                       # OpenCV pads both axes when either needs it
        eh, ew = h + (4 - h % 4), w + (4 - w % 4)
    return eh // 4, ew // 4


def _tile_pair(coord, t):
    tf = np.float32(np.float32(coord) * (np.float32(1) / np.float32(t))) - np.float32(0.5)
    t1 = int(math.floor(tf))
    return max(t1, 0), min(t1 + 1, 3)


def _axis_ok(n0, span, first, last, n, t):
    pairs = [_tile_pair(_reflect101(n0 + k - 3, n), t) for k in range(span)]
    a, b = _tile_pair(_reflect101(n0 + first, n), t), _tile_pair(_reflect101(n0 + last, n), t)
    return all(p == a or p == b for p in pairs)


def packed_tiles(h, w):
    """bool [tiles y, tiles x]: True where k_prefilter takes the packed CLAHE path (at most two CLAHE tile pairs per axis)."""
    th, tw = clahe_geom(h, w)
    ok_x = np.array([_axis_ok(x0, PF_TW + 8, -3, PF_TW + 4, w, tw) for x0 in range(0, w, PF_TW)])
    ok_y = np.array([_axis_ok(y0, PF_TH + 6, -3, PF_TH + 2, h, th) for y0 in range(0, h, PF_TH)])
    return ok_y[:, None] & ok_x[None, :]


# ------------------------------------------------------------------------------------------------
# inputs
# ------------------------------------------------------------------------------------------------
PRODUCTION = [(2160, 3840), (1080, 1920), (2160, 960)]          # 4K luma, 1080p luma = the (2,2) chroma of 4K, the (1,4) chroma of 4K
PADDING = [(1080 + a, 1920 + b) for a in range(4) for b in range(4) if a or b] + [(2161, 3839)]   # every nonzero (h % 4, w % 4)
REGIME_SWEEP = [(h, w) for h in (272, 277, 280, 283, 288) for w in (532, 537, 540, 543, 546, 552)]
SEAM_W = [1, 2, 3, 4, 5, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 513]
SEAM_H = [1, 2, 3, 5, 31, 32, 33, 63, 64, 65, 70, 71]
SEAMS = ([(h, w) for w in SEAM_W for h in (1, 33, 70)] + [(h, w) for h in SEAM_H for w in (1, 65, 300)] + [(7, 4096), (4095, 5)])
SEAMS = sorted(set(SEAMS))
KINDS = ["noise", "vignette", "levels5", "steps60", "flat", "checker", "blocks", "ramp22", "ramp67"]
CANNY_THR = [(0.0, 0.0), (5.0, 200.0), (200.0, 5.0), (90.0, 90.0), (50.5, 60.25), (100.0, 32767.0), (40000.0, 50000.0)]


def plane(kind, h, w, seed=0):
    rng = np.random.default_rng([seed, h, w])
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == "noise":                    # every LUT entry, the bilateral redo and many ties
        return rng.integers(0, 256, (h, w), dtype=np.uint8)
    if kind == "vignette":                 # noise whose range grows across the plane: CLAHE tiles with very different LUTs
        return (rng.integers(0, 256, (h, w)) * (yy + xx + 1) // (h + w)).astype(np.uint8)
    if kind == "levels5":                  # few-level plane (JzAzBz-like luma): CLAHE clipping
        return rng.integers(0, 5, (h, w), dtype=np.uint8)
    if kind == "steps60":                  # {0, 60, .., 240} in 7 x 13 blocks: large gradients
        blk = rng.integers(0, 5, (h // 7 + 1, w // 13 + 1)) * 60
        return blk[yy // 7, xx // 13].astype(np.uint8)
    if kind == "flat":                     # all mass in one bin: the residual redistribution
        return np.full((h, w), 77, np.uint8)
    if kind == "checker":                  # period-1 checkerboard: the largest magnitudes
        return (((yy + xx) & 1) * 255).astype(np.uint8)
    if kind == "blocks":                   # 0 / 255 blocks
        blk = rng.integers(0, 2, (h // 16 + 1, w // 16 + 1)) * 255
        return blk[yy // 16, xx // 16].astype(np.uint8)
    if kind == "ramp22":                   # gradient ratio 5/12 ~ tan 22.5: both sides of the class boundary
        return ((12 * xx + 5 * yy) // 4 % 256).astype(np.uint8)
    if kind == "ramp67":
        return ((5 * xx + 12 * yy) // 4 % 256).astype(np.uint8)
    raise ValueError(kind)


# ------------------------------------------------------------------------------------------------
# CPU self-checks of the references
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(1080, 1920), (1081, 1917), (283, 537), (70, 257), (7, 4096), (4095, 5), (1, 33), (2, 2)])
def test_references_agree_with_oracle(cv, shape):
    for kind in ("noise", "levels5", "checker", "ramp22"):
        p = plane(kind, *shape, seed=1)
        cl = ref_clahe(p)
        assert np.array_equal(cl, O.clahe(p)), (kind, "CLAHE " + first_diff(cl, O.clahe(p)))
        g = ref_gauss(cl)
        assert np.array_equal(g, O.gauss3(cl)), (kind, "Gaussian")
        b = O.bilateral5(g)
        lo, hi = ref_thresholds(b)
        assert O.percentile_thresholds(b) == (lo, hi), (kind, "thresholds")
        for t in [(lo, hi)] + CANNY_THR:
            assert np.array_equal(ref_canny(b, *t), O.canny_u8(b, *t) == 1), (kind, t, "Canny")
        layer = (p.astype(np.float32) / np.float32(255)).astype(np.float32)
        assert np.array_equal(ref_chain(layer), O.canny(layer) == 1), (kind, "chain")


@pytest.mark.parametrize("shape,kind", [((1080, 1920), "noise"), ((1081, 1917), "levels5"), ((540, 960), "ramp22"), ((33, 70), "noise")])
def test_bilateral64_tie_band_holds_for_opencv_and_oracle(cv, shape, kind):
    g = ref_gauss(ref_clahe(plane(kind, *shape, seed=2)))
    q = ref_bilateral64(g)
    n = check_tie_band(O.bilateral5(g), q)
    check_tie_band(cv.bilateralFilter(g, 5, 75, 75), q)
    print(f"bilateral64 {shape} {kind}: {n} px within {TIE_BAND} of a tie")


def test_regime_sweep_straddles_the_packed_boundary():
    """The sweep contains planes whose prefilter tiles all take the packed path, planes with general tiles, and planes with
    tiles of both kinds side by side; production sizes take the packed path everywhere."""
    kinds = [packed_tiles(h, w) for h, w in REGIME_SWEEP]
    assert any(k.all() for k in kinds)
    assert any(not k.any() for k in kinds) or any((~k).any() for k in kinds)
    assert any(k.any() and not k.all() for k in kinds), "no plane mixes packed and general tiles"
    for h, w in PRODUCTION + PADDING:
        assert packed_tiles(h, w).all(), (h, w)
    assert not packed_tiles(144, 256).any()       # the size of the older stage tests: general path only


# ------------------------------------------------------------------------------------------------
# GPU: every stage call at production sizes, padding, regime boundary and seams
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def st():
    from aeaj.codec import get_stages
    return get_stages(0)


def check_stages(st, p, bil64=False, thr=()):
    """Each stage on the reference output of the previous one; returns the tie-band count (None without bil64)."""
    cl = ref_clahe(p)
    got = st.clahe(p)
    assert np.array_equal(got, cl), "CLAHE: " + first_diff(got, cl)
    g = ref_gauss(cl)
    got = st.gauss3(cl)
    assert np.array_equal(got, g), "Gaussian: " + first_diff(got, g)
    b = O.bilateral5(g)
    got = st.bilateral5(g)
    assert np.array_equal(got, b), "bilateral vs the oracle: " + first_diff(got, b)
    n = check_tie_band(got, ref_bilateral64(g)) if bil64 else None
    lo, hi = ref_thresholds(b)
    assert st.percentile_thresholds(b) == (lo, hi), "percentile thresholds"
    for t in [(lo, hi)] + list(thr):
        got = st.canny_u8(b, *t) == 1
        assert np.array_equal(got, ref_canny(b, *t)), f"Canny {t}: " + first_diff(got, ref_canny(b, *t))
    layer = (p.astype(np.float32) / np.float32(255)).astype(np.float32)
    got = st.canny(layer) == 1
    assert np.array_equal(got, ref_chain(layer)), "whole chain: " + first_diff(got, ref_chain(layer))
    return n


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", PRODUCTION)
def test_stages_production(cv, st, shape, kind):
    bil64 = kind in ("noise", "levels5", "ramp22") or shape[0] * shape[1] <= 1080 * 1920
    n = check_stages(st, plane(kind, *shape, seed=3), bil64=bil64, thr=CANNY_THR if kind == "noise" else ())
    if n is not None:
        print(f"\n{shape} {kind}: {n} px within {TIE_BAND} of a bilateral tie")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", PADDING)
def test_stages_clahe_padding(cv, st, shape):
    check_stages(st, plane("noise", *shape, seed=4))
    check_stages(st, plane("steps60", *shape, seed=4))


@pytest.mark.gpu
def test_stages_halo_split_size(cv, st):
    """One 8192 x 8192 plane, the size the halo split is for, against the oracle and cv2."""
    check_stages(st, plane("noise", 8192, 8192, seed=5))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", REGIME_SWEEP)
def test_stages_regime_boundary(cv, st, shape):
    for kind in ("noise", "ramp67"):
        check_stages(st, plane(kind, *shape, seed=6), bil64=True)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SEAMS)
def test_stages_tile_seams(cv, st, shape):
    for kind in ("noise", "levels5", "blocks"):
        check_stages(st, plane(kind, *shape, seed=7), bil64=True, thr=CANNY_THR[:4])


# ------------------------------------------------------------------------------------------------
# GPU: hysteresis stress at 2160 x 3840 (canny_u8 against cv2.Canny)
# ------------------------------------------------------------------------------------------------
H4K, W4K = 2160, 3840


def tile_links(e):
    """8-neighbour pairs of edge pixels in different hysteresis tiles -> (corner links, other links)"""
    h, w = e.shape
    corner = other = 0
    for dy, dx in ((0, 1), (1, 0), (1, 1), (1, -1)):
        a = e[:h - dy, max(0, -dx):w - max(0, dx)]
        b = e[dy:, max(0, dx):w - max(0, -dx)]
        y0, x0 = np.nonzero(a & b)
        x0 = x0 + max(0, -dx)
        cy, cx = (y0 // HY_TH) != ((y0 + dy) // HY_TH), (x0 // HY_TW) != ((x0 + dx) // HY_TW)
        corner += int((cy & cx).sum())
        other += int((cy ^ cx).sum())
    return corner, other


def serpentine():
    img = np.zeros((H4K, W4K), np.uint8)
    ys = list(range(10, H4K - 14, 12))
    for k, y in enumerate(ys):
        img[y:y + 3, 10:W4K - 10] = 120
        if k + 1 < len(ys):
            x = W4K - 13 if k % 2 == 0 else 10
            img[y:y + 15, x:x + 3] = 120
    y = ys[-1]
    x = 10 if len(ys) % 2 == 0 else W4K - 40
    img[y:y + 3, x:x + 30] = 255                          # the seed: far end of the chain, last hysteresis tile row
    return img


def spiral():
    img = np.zeros((H4K, W4K), np.uint8)
    t, l, b, r = 10, 10, H4K - 13, W4K - 13
    last = None
    while b - t > 24 and r - l > 24:
        img[t:t + 3, l:r + 3] = 120                       # top, left to right
        img[t:b + 3, r:r + 3] = 120                       # right, down
        img[b:b + 3, l + 12:r + 3] = 120                  # bottom, right to left
        img[t + 12:b + 3, l + 12:l + 15] = 120            # left, up to the next turn
        last = (t + 12, l + 12)
        t, l, b, r = t + 12, l + 12, b - 12, r - 12
    img[last[0]:last[0] + 3, last[1]:last[1] + 30] = 255  # seed at the centre: propagation runs outwards in all directions
    return img


def staircase(anti):
    """Step edges along lines of slope 1/8 through hysteresis tile corners (32 rows per 256 columns): the edge runs cross
    tiles only diagonally at a corner, and cross bitmap words inside a tile (bit 31 -> bit 0).  Stripes of 64 rows
    alternate 0 / 100 (weak edges); the bright pixels of the 16 columns where the lines end lowest are 250 (strong seeds),
    so propagation climbs through up-left (diag) or up-right (anti) tile corners."""
    yy, xx = np.mgrid[0:H4K, 0:W4K]
    xs = (W4K - 1 - xx) if anti else xx
    img = np.where(((yy - (xs - 1) // 8 - 1) // 64) % 2 == 1, 100, 0).astype(np.uint8)
    img[(xs >= W4K - 16) & (img == 100)] = 250
    return img


STRESS = {"serpentine": (serpentine, [(5.0, 200.0), (100.0, 600.0)]),
          "spiral": (spiral, [(5.0, 200.0), (100.0, 600.0)]),
          "staircase_diag": (lambda: staircase(False), [(300.0, 800.0)]),
          "staircase_anti": (lambda: staircase(True), [(300.0, 800.0)])}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(STRESS))
def test_hysteresis_stress(cv, st, name):
    make, thrs = STRESS[name]
    img = make()
    for lo, hi in thrs:
        want = ref_canny(img, lo, hi)
        weak_or_strong = ref_canny(img, lo, lo)
        assert want.sum() > 0.85 * weak_or_strong.sum(), "the pattern must be reached from its seeds"
        if name.startswith("staircase"):
            corner, other = tile_links(want[:, HY_TW:-HY_TW])           # the seed columns are left out
            assert corner > 100 and other == 0, (corner, other)
        got = st.canny_u8(img, lo, hi) == 1
        assert np.array_equal(got, want), f"{name} {lo, hi}: " + first_diff(got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("lo", [110.0, 130.0, 150.0])
def test_hysteresis_percolation(cv, st, lo):
    """Blurred noise with lo near the 8-connected percolation point of its weak pixels: one huge fractal cluster."""
    p = ref_gauss(plane("noise", H4K, W4K, seed=8))
    want = ref_canny(p, lo, 500.0)
    got = st.canny_u8(p, lo, 500.0) == 1
    print(f"\npercolation lo={lo}: {want.mean():.3f} of the pixels are edges")
    assert np.array_equal(got, want), first_diff(got, want)


# ------------------------------------------------------------------------------------------------
# GPU: the fused batch path, mixed content
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def codec():
    from aeaj.codec import get_codec
    return get_codec(0)


def frames(h, w):
    """noise, synth, few-level and flat RGB frames, float32 k/255.  The noise is mid-range (100 .. 199, a little colour) with
    15 % of 32 x 32 blocks dark: the percentile thresholds then fall far apart, strong pixels sit on the block borders only,
    and most edges are weak pixels reached through long chains -- the load that keeps the hysteresis queue busy."""
    rng = np.random.default_rng([9, h, w])
    yy, xx = np.mgrid[0:h, 0:w]
    dark = (rng.random((h // 32 + 1, w // 32 + 1)) < 0.15)[yy // 32, xx // 32]
    noise = np.where(dark, 10, rng.integers(100, 200, (h, w)))[..., None] + rng.integers(-6, 7, (h, w, 3))
    few = (rng.integers(0, 3, (h // 9 + 1, w // 9 + 1, 3)) * 127)[yy // 9, xx // 9]
    out = [np.clip(noise, 0, 255), np.round(synth(h, w, seed=9) * 255), few, np.full((h, w, 3), 128)]
    return np.stack([(f.astype(np.float32) / np.float32(255)).astype(np.float32) for f in out])


FUSED_SHAPES = [(2160, 3840), (1081, 1917), (283, 537), (67, 130)]


@pytest.mark.gpu
def test_fused_batch_edges(cv, codec):
    """Every image and layer of a mixed batch equals the reference chain on the GPU's own layer (exact even in the PQ spaces)
    and the same frame encoded alone; at least one batch needs more hysteresis re-visits than it has tiles."""
    import torch
    ratios = []
    for space, (H, W) in [(sp, shape) for sp in ("YCbCr", "ICtCp", "JzAzBz") for shape in FUSED_SHAPES]:
        rgb = frames(H, W)
        B = len(rgb)
        enc = codec.encode(torch.from_numpy(rgb).cuda(), space, (30, 95), (4, 64), taps=True)
        status = enc.status[:2].cpu().numpy()
        layers = [t.cpu().numpy() for t in enc.layers]
        edges = [t.cpu().numpy() for t in enc.edges]
        assert status[1] == 1, f"{space} {H}x{W}: hysteresis did not converge"
        ntiles = B * sum(math.ceil(math.ceil(e.shape[2] / 32) / 8) * math.ceil(e.shape[1] / HY_TH) for e in edges)
        ratios.append(int(status[0]) / ntiles)
        print(f"\n{space} {H}x{W} B={B}: {int(status[0])} hysteresis re-visits over {ntiles} tiles")
        for b in range(B):
            for l in range(3):
                want = ref_chain(layers[l][b])
                assert np.array_equal(edges[l][b] == 1, want), f"{space} {H}x{W} image {b} layer {l}: " + first_diff(edges[l][b] == 1, want)
        for b in range(B):
            one = codec.encode(torch.from_numpy(rgb[b:b + 1]).cuda(), space, (30, 95), (4, 64), taps=True)
            for l in range(3):
                e1 = one.edges[l][0].cpu().numpy()
                assert np.array_equal(e1, edges[l][b]), f"{space} {H}x{W} image {b} layer {l}: B = {B} and B = 1 differ"
    assert max(ratios) > 1.0, f"the work queue was never exercised beyond one pass per tile: {ratios}"


# ------------------------------------------------------------------------------------------------
# stage calls reject pointers the kernels cannot use
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_stage_calls_reject_misaligned_pointers(st):
    import ctypes as C
    import torch
    lib, hd = st.lib, st.handle
    EINVAL = -1
    h, w = 64, 128
    sentinel = 0xAB
    src = torch.randint(0, 256, (h * w + 16,), dtype=torch.uint8, device="cuda")
    dst = torch.full((h * w + 16,), sentinel, dtype=torch.uint8, device="cuda")
    layer = torch.rand(h * w + 4, device="cuda")
    thr = torch.tensor([10.0, 20.0], dtype=torch.float64, device="cuda")
    mn, mx = 4, 64
    ws = torch.empty(int(lib.aeaj_stage_workspace_bytes(h, w, mn, mx)) + 512, dtype=torch.uint8, device="cuda")
    leaves = torch.zeros((1024, 4), dtype=torch.int32, device="cuda")
    states = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    counts = torch.zeros(4, dtype=torch.int32, device="cuda")
    coef = torch.zeros(h * w, dtype=torch.int32, device="cuda")
    qtab = (C.c_void_p * 9)()
    S, D, L, T, WS = src.data_ptr(), dst.data_ptr(), layer.data_ptr(), thr.data_ptr(), ws.data_ptr()
    s = torch.cuda.current_stream().cuda_stream
    assert S % 256 == 0 and D % 256 == 0 and WS % 256 == 0
    calls = []
    for fn in (lib.aeaj_clahe, lib.aeaj_gauss3, lib.aeaj_bilateral5):
        for a, b, c in ((S + 1, D, WS), (S + 2, D, WS), (S, D + 1, WS), (S, D + 3, WS), (S, D, WS + 1), (S, D, WS + 16), (S, D, WS + 128)):
            calls.append((fn, (hd, a, h, w, b, c, s)))
    for a, e, c in ((S + 1, D, WS), (S, D + 2, WS), (S, D, WS + 4)):
        calls.append((lib.aeaj_canny_u8, (hd, a, h, w, T, e, c, s)))
    calls += [(lib.aeaj_canny, (hd, L + 2, h, w, D, WS, s)), (lib.aeaj_canny, (hd, L, h, w, D, WS + 64, s)),
              (lib.aeaj_percentile_thresholds, (hd, S, h, w, T, WS + 8, s)),
              (lib.aeaj_quadtree, (hd, S, h, w, mn, mx, leaves.data_ptr(), states.data_ptr(), counts.data_ptr(), WS + 32, s)),
              (lib.aeaj_dct_quant, (hd, L, h, w, 0.5, 1.0, leaves.data_ptr(), counts.data_ptr(), mn, mx, qtab, coef.data_ptr(), WS + 1, s)),
              (lib.aeaj_dequant_idct, (hd, coef.data_ptr(), leaves.data_ptr(), counts.data_ptr(), mn, mx, qtab, h, w, 0.5, 1.0, L, WS + 1, s))]
    for fn, args in calls:
        assert fn(*args) == EINVAL, (fn.__name__, args)
        assert b"aligned" in lib.aeaj_last_error(), lib.aeaj_last_error()
    torch.cuda.synchronize()
    assert bool((dst == sentinel).all()), "a rejected call wrote its output"
    assert lib.aeaj_clahe(hd, S, h, w, D, WS, s) == 0                  # aligned pointers still run
    torch.cuda.synchronize()
    assert np.array_equal(dst[:h * w].cpu().numpy().reshape(h, w), O.clahe(src[:h * w].cpu().numpy().reshape(h, w)))
