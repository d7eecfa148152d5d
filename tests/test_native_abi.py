"""CPU-side checks of the product's host logic and of the C-ABI boundary (no compute calls)."""
import ctypes
import hashlib
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from aeaj import native
    lib = native.load()
    hdr = open(os.path.join(ROOT, "include", "aeaj.h")).read()
    declared = sorted(set(re.findall(r"AEAJ_API[^;]*?\b(aeaj_\w+)\s*\(", hdr)))
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/aeaj.h but not exported"
    assert sorted(native.EXPORTS) == declared
    assert lib.aeaj_version() == 3


def test_no_cpu_fallback_without_cuda():
    import torch
    from aeaj import native
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    lib = native.load()
    h = ctypes.c_void_p()
    rc = lib.aeaj_create(0, ctypes.byref(h))
    assert rc == -3 and b"no CPU fallback" in lib.aeaj_last_error()        # AEAJ_ENOCUDA
    from color import convert
    with pytest.raises(native.AeajError):
        convert("sRGB", "YCbCr", np.zeros((4, 3), np.float32))
    from image import Image
    from jpeg import Jpeg, JpegCompressionSettings
    with pytest.raises(native.AeajError):
        Jpeg(JpegCompressionSettings()).compress(Image.from_array(np.zeros((8, 8, 3), np.float32)))


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "adaptive-edge-aware-jpeg_b200")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(d, f)).read()
                assert "import oracle" not in src and "aeaj_oracle" not in src and "ref_import" not in src, f


def test_host_tables_match_reference_golden(golden):
    from aeaj import tables as T
    sha = lambda a: hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()
    for key, want in golden.meta["qmatrix_sha"].items():
        t, size = key.split("_")
        base = T.LUMINANCE_Q if t == "luma" else T.CHROMINANCE_Q
        allq = np.stack([T.quantization_matrix(base, int(size), q) for q in range(1, 100)]).astype(np.int32)
        assert sha(allq) == want, key
    assert golden.meta["qmatrix_sha_modeD_equal"] is True       # q tables do not depend on the IPP switch
    for key, want in golden.meta["quality_factor"].items():
        bmin, bmax, qmin, qmax = map(int, key.split(","))
        assert [T.quality_factor(s, (qmin, qmax), (bmin, bmax)) for s in T.block_sizes((bmin, bmax))] == want
    for s, want in golden.meta["zigzag_sha"].items():
        assert sha(T.zigzag_ordering(int(s))) == want
    assert T.layer_shapes(135, 241, "ICtCp") == [(135, 241), (135, 60), (135, 60)]
    assert T.layer_shapes(135, 241, "YCbCr") == [(135, 241), (67, 120), (67, 120)]


def test_settings_and_shim_surface_without_gpu():
    from jpeg import Jpeg, JpegCompressionSettings
    from jpeg.utils import largest_power_of_2
    from color import get_color_spaces
    s = JpegCompressionSettings()
    assert (s.color_space, s.quality_range, s.block_size_range) == ("YCoCg", (40, 80), (4, 64))
    assert s.downsampling_ratios.tolist() == [[1, 1], [2, 2], [2, 2]]
    assert JpegCompressionSettings("ICtCp").downsampling_ratios.tolist() == [[1, 1], [1, 4], [1, 4]]
    with pytest.raises(ValueError):
        JpegCompressionSettings("XYZ")
    j = Jpeg(JpegCompressionSettings("YCbCr", (50, 90), (4, 64)))
    assert [j._get_quality_factor(k) for k in (4, 8, 16, 32, 64)] == [90, 80, 70, 60, 50]
    j.update_layer_shapes((2160, 3840))
    assert j.layer_shapes.tolist() == [[2160, 3840], [1080, 1920], [1080, 1920]]
    assert [largest_power_of_2(n) * 2 for n in (1, 2, 3, 4, 5, 512, 513, 1080, 3840, 8192)] == [2, 4, 4, 4, 8, 512, 1024, 2048, 4096, 8192]
    with pytest.raises(ValueError):
        largest_power_of_2(0)
    assert len(get_color_spaces()) == 7


def test_host_state_helpers_round_trip():
    import oracle as O
    from aeaj import native
    lib = native.load()
    rng = np.random.default_rng(0)
    for shape, (mn, mx) in [((130, 257), (4, 64)), ((33, 17), (2, 128)), ((4, 4), (4, 64)), ((511, 513), (8, 32))]:
        edge = (rng.random(shape) < 0.01).astype(np.float32)
        leaves, states, root = O.quadtree(edge, mx, mn)
        got, ncoef = native.states_to_leaves(states, root, *shape)
        assert np.array_equal(got[:, :3], leaves) and ncoef == int((leaves[:, 2].astype(np.int64) ** 2).sum())
        packed = np.empty((len(states) + 3) // 4, dtype=np.uint8)
        assert lib.aeaj_pack_states_host(states.ctypes.data, len(states), packed.ctypes.data) == 0
        assert packed.tobytes() == O.pack_states(states)


def test_corrupt_state_streams_are_rejected():
    """The state stream of an .ajpg file is untrusted input (ADVICE r1): a wrong root, a leaf outside the block range or the
    layer, or a split below size 2 must raise instead of reaching the device (the reference dies with a KeyError there)."""
    import oracle as O
    from aeaj import native
    rng = np.random.default_rng(1)
    shape, (mn, mx) = (130, 257), (4, 64)
    edge = (rng.random(shape) < 0.01).astype(np.float32)
    leaves, states, root = O.quadtree(edge, mx, mn)
    got, _ = native.states_to_leaves(states, root, *shape, (mn, mx))
    assert np.array_equal(got[:, :3], leaves)
    with pytest.raises(ValueError):                                    # root taken "straight from the stream"
        native.states_to_leaves(states, root * 2, *shape, (mn, mx))
    with pytest.raises(ValueError):                                    # a leaf of the root's size (512 > block_max)
        native.states_to_leaves(np.array([0], np.uint8), root, *shape, (mn, mx))
    with pytest.raises(ValueError):                                    # splits all the way down: size 1, then 0
        native.states_to_leaves(np.ones(64, np.uint8), 4, 3, 3, (2, 2))
    with pytest.raises(ValueError):                                    # leaves below block_min
        native.states_to_leaves(np.array([1, 1, 0, 0, 0, 0, 0, 0, 0], np.uint8), 8, 8, 8, (4, 8))
    bad = states.copy()
    k = int(np.nonzero(bad == 2)[0][0])                                # an out-of-bounds node declared a leaf
    bad[k] = 0
    with pytest.raises(ValueError):
        native.states_to_leaves(bad, root, *shape, (mn, mx))
    # a truncated stream yields the leaves seen so far (jpeg.py:784 stops the same way); the caller's length check catches it
    part, _ = native.states_to_leaves(states[: len(states) // 2], root, *shape, (mn, mx))
    assert 0 < len(part) < len(leaves)


def test_packed_coefficient_host_helpers():
    """aeaj_pack_coefficients_host / aeaj_unpack_coefficients_host: the packed PCIe form (bit mask + int16 non-zeros)"""
    from aeaj import native
    rng = np.random.default_rng(0)
    for n in (0, 1, 31, 32, 33, 1000, 100003):
        c = (rng.integers(-300, 300, n) * (rng.random(n) < 0.2)).astype(np.int32)
        m, v, ovf = native.pack_coefficients_host(c)
        assert not ovf and m.size == (n + 31) // 32 and v.size == int((c != 0).sum())
        assert np.array_equal(native.unpack_coefficients_host(m, v, n), c)
    assert native.pack_coefficients_host(np.array([0, 40000, -5], np.int32))[2]           # does not fit int16: flagged
    m, v, _ = native.pack_coefficients_host(np.array([1, 0, 2, 0, 0, 3], np.int32))
    with pytest.raises(ValueError):
        native.unpack_coefficients_host(m, v[:2], 6)                                         # fewer values than mask bits
    with pytest.raises(ValueError):
        native.unpack_coefficients_host(m[:0], v, 6)                                         # mask too short
