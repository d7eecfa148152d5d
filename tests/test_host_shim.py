"""CPU tests of the host-side shim logic that needs no GPU: the Image container (image/image.py:26-149 semantics plus the
8-bit source shortcut), .ajpg framing helpers and the error behaviour of the drop-in classes."""
import os

import numpy as np
import pytest

from image import Image
from jpeg import Jpeg, JpegCompressionSettings


def _px(h=6, w=5, seed=0):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)


def test_image_from_uint8_matches_load_semantics():
    px = _px()
    img = Image.from_uint8(px, ".png")
    assert img.uint8_source() is px or np.array_equal(img.uint8_source(), px)
    assert img.ndim == 3 and img.original_shape == px.shape
    assert np.array_equal(img.get_uint8(), ((px.astype(np.float32) / 255.0) * 255).astype(np.uint8))   # image.py:84 then :127
    ref = px.astype(np.float32) / 255.0                       # what Image.load produces (image.py:84)
    data = img.data
    assert data.dtype == np.float32 and np.array_equal(data, ref)
    assert img.uint8_source() is None                         # the floats were handed out: no shortcut any more
    data[0, 0, 0] = 0.25                                      # ... because the caller may now change them
    assert img.data[0, 0, 0] == np.float32(0.25)


def test_image_data_assignment_and_copy_and_reshape():
    px = _px(4, 4, 1)
    img = Image.from_uint8(px)
    cp = img.copy()
    assert cp.uint8_source() is not None and cp.uint8_source() is not img.uint8_source()
    img.reshape((16, 3))
    assert img.uint8_source().shape == (16, 3) and img.ndim == 2
    img.data = np.zeros((4, 4, 3), np.float32)
    assert img.uint8_source() is None and img.ndim == 3
    flat = Image.from_array(np.ones((2, 3, 3), np.float32)).get_flattened()
    assert flat.shape == (6, 3)
    with pytest.raises(ValueError):
        Image.from_uint8(np.zeros((4, 4), np.uint8))
    with pytest.raises(ValueError):
        Image.from_uint8(np.zeros((4, 4, 3), np.float32))


def test_compress_argument_checks_need_no_gpu():
    j = Jpeg(JpegCompressionSettings("YCbCr", (30, 95), (4, 64)))
    with pytest.raises(TypeError):
        j.compress(np.zeros((4, 4, 3), np.float32))           # jpeg.py:250-251
    with pytest.raises(ValueError):
        j.compress(Image.from_array(np.zeros((16, 3), np.float32)))   # jpeg.py:252-253
    with pytest.raises(ValueError):
        JpegCompressionSettings("NoSuchSpace")                 # jpeg.py:164-165


def test_state_stream_parse_rejects_truncated_coefficients():
    """_entropy_decode cross-checks the inflated coefficient length against the quadtree header."""
    import json, zlib
    meta = {"height": 8, "width": 8, "num_layers": 1, "color_space": "YCbCr", "quality_min": 30, "quality_max": 95,
            "block_size_min": 4, "block_size_max": 8, "extension": ".png"}
    mb = json.dumps(meta).encode()
    states = bytes([0b00000000])                               # one leaf of the 8x8 root: '00'
    body = (2).to_bytes(4, "big") + (8).to_bytes(4, "big") + states
    coef = zlib.compress(np.zeros(10, np.int32).tobytes())     # 10 != 64 coefficients
    blob = len(mb).to_bytes(4, "big") + mb + body + len(coef).to_bytes(4, "big") + coef
    with pytest.raises(ValueError):
        Jpeg(JpegCompressionSettings())._entropy_decode(blob)


def test_evaluation_metrics_surface_and_known_answers():
    """EvaluationMetrics(original, compressed).psnr() / .ssim() / .ms_ssim() (evaluation_metrics.py:31-110): piq's published
    formulas restated with torch; known answers that do not need piq."""
    import torch
    from image import EvaluationMetrics
    from image.evaluation_metrics import rgb_to_gray_u8
    rng = np.random.default_rng(0)
    a = rng.random((200, 240, 3), dtype=np.float32)
    img_a, img_same = Image.from_array(a.copy()), Image.from_array(a.copy())
    ev = EvaluationMetrics(img_a, img_same)
    assert isinstance(ev.psnr(), torch.Tensor) and abs(float(ev.psnr()) - 80.0) < 1e-3        # -10 log10(0 + 1e-8)
    assert abs(float(ev.ssim()) - 1.0) < 1e-6 and abs(float(ev.ms_ssim()) - 1.0) < 1e-5
    b = np.clip(a * 0.0 + 0.5, 0, 1).astype(np.float32)
    c = (b + 0.1).astype(np.float32)                                                          # mse = 0.01 -> 20 dB
    assert abs(float(EvaluationMetrics(Image.from_array(b), Image.from_array(c)).psnr()) - 20.0) < 1e-3
    noisy = np.clip(a + rng.normal(0, 0.1, a.shape).astype(np.float32), 0, 1)
    s1 = float(EvaluationMetrics(img_a, Image.from_array(noisy)).ssim())
    s2 = float(EvaluationMetrics(Image.from_array(noisy), img_a).ssim())
    assert 0.0 < s1 < 0.99 and abs(s1 - s2) < 1e-6                                            # symmetric, penalises noise
    m = float(EvaluationMetrics(img_a, Image.from_array(noisy)).ms_ssim())
    assert 0.0 < m < 1.0
    with pytest.raises(ValueError):
        EvaluationMetrics(Image.from_array(a[:100, :100].copy()), Image.from_array(a[:100, :100].copy())).ms_ssim()
    with pytest.raises(NotImplementedError):
        ev.lpips()
    with pytest.raises(TypeError):
        EvaluationMetrics._image_to_tensor([1, 2, 3])
    # the reference's grey conversion: cv2.cvtColor(rgb, cv2.COLOR_RGB2GRAY) of OpenCV 4.13, stored for 64 x 48 random pixels
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gray_u8.npz"))
    assert np.array_equal(rgb_to_gray_u8(g["rgb"]), g["gray"])
