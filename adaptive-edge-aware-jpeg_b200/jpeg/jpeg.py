"""Jpeg / JpegCompressionSettings drop-in (src/jpeg/jpeg.py:36-800).

``compress`` / ``decompress`` keep the reference's signatures, exceptions and the byte-compatible
.ajpg container (jpeg.py:531-674); everything between the colour transform and the quantised
coefficients -- and back -- runs on the GPU through libaeaj.so (aeaj_encode / aeaj_decode).
Entropy coding (zigzag gather, state packing, zlib level 9) stays on the host, as in the reference -- unless
``Jpeg(settings, deflate="device")`` selects the device coder and decoder: compress writes valid zlib streams that are not
zlib's bytes, decompress inflates any .ajpg file's streams on the GPU.
``compress_batch`` / ``decompress_batch`` are additions for same-shape batches.
"""
from __future__ import annotations

import json
import os
import zlib
from concurrent.futures import ThreadPoolExecutor
from io import BytesIO
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from aeaj import native, tables
from aeaj.codec import get_codec
from image import Image


class JpegCompressionSettings:
    """Compression parameters (jpeg.py:36-174)."""

    LUMINANCE_QUANTIZATION_MATRIX = tables.LUMINANCE_Q
    CHROMINANCE_QUANTIZATION_MATRIX = tables.CHROMINANCE_Q
    COLOR_SPACE_SETTINGS = {
        name: {
            "downsampling_ratios": np.array([[1, 1], list(tables.CHROMA_SUBSAMPLING[name]), list(tables.CHROMA_SUBSAMPLING[name])]),
            "quantization_matrices": [tables.LUMINANCE_Q, tables.CHROMINANCE_Q, tables.CHROMINANCE_Q],
        }
        for name in tables.CODEC_SPACES
    }

    def __init__(self, color_space: str = "YCoCg", quality_range: Tuple[int, int] = (40, 80),
                 block_size_range: Tuple[int, int] = (4, 64)) -> None:
        if color_space not in self.COLOR_SPACE_SETTINGS:
            raise ValueError(f"Unsupported color space: {color_space}")
        self.color_space = color_space
        self.quality_range = quality_range
        self.block_size_range = block_size_range
        cfg = self.COLOR_SPACE_SETTINGS[color_space]
        self.downsampling_ratios: np.ndarray = cfg["downsampling_ratios"]
        self.quantization_matrices: List[np.ndarray] = cfg["quantization_matrices"]


def _zigzag_stream(coef: np.ndarray, sizes: np.ndarray, zz_cache: dict, inverse: bool) -> np.ndarray:
    """Per-block zigzag gather (jpeg.py:579-585) / scatter (jpeg.py:664-672) on the concatenated
    coefficient stream, vectorised per size class."""
    out = np.empty_like(coef)
    sizes = sizes.astype(np.int64)
    offs = np.concatenate([[0], np.cumsum(sizes * sizes)])
    for s in np.unique(sizes):
        idx = np.nonzero(sizes == s)[0]
        zz = zz_cache[int(s)].astype(np.int64)
        base = offs[idx][:, None]
        lin = (base + np.arange(s * s)[None, :]).ravel()
        per = (base + zz[None, :]).ravel()
        if inverse:
            out[per] = coef[lin]
        else:
            out[lin] = coef[per]
    return out


def _raise_inflate_status(status: np.ndarray) -> None:
    """the first failed plane of aeaj_inflate_coefficients as the host path's exception: ValueError for a length mismatch
    (as its size check), zlib.error for everything else"""
    from aeaj.codec import INFLATE_ERRORS, INFLATE_LENGTH
    for code in status.ravel():
        if code == INFLATE_LENGTH:
            raise ValueError(INFLATE_ERRORS[INFLATE_LENGTH])
        if code:
            raise zlib.error(f"Error while decompressing data on the device: {INFLATE_ERRORS.get(int(code), int(code))}")


class Jpeg:
    """Adaptive-block JPEG codec (jpeg.py:177-800) backed by the B200 hot path."""

    def __init__(self, settings: JpegCompressionSettings, deflate: str = "host") -> None:
        """deflate: where the zlib layer of the coefficient streams runs, in both directions.
        "host" (default): compress codes them with zlib level 9, the reference's own bytes; decompress uses zlib.decompress.
        "device": compress deflates them on the GPU (aeaj_deflate_coefficients) and moves only the compressed bytes -- faster
        end to end and about 15 % larger (DESIGN.md section 5), readable by every .ajpg decoder, the reference's included, but
        not byte-identical to its files; decompress inflates them on the GPU (aeaj_inflate_coefficients), straight into the
        buffers the decoder reads.  It reads any .ajpg file, the reference's zlib-9 files included, and gives the same images.
        Errors: a corrupt zlib section raises zlib.error and a coefficient count that does not match the quadtree header raises
        ValueError, as on the host -- with one difference: a stream that inflates past the expected length raises ValueError
        even where zlib.decompress would have met a later error in it first."""
        if deflate not in ("host", "device"):
            raise ValueError("deflate must be 'host' or 'device'")
        self.deflate = deflate
        self.update_settings(settings)

    # -- settings / caches ----------------------------------------------------------------------
    def update_settings(self, settings: JpegCompressionSettings, layer_shape: Optional[Tuple[int, int]] = None) -> None:
        self.settings = settings
        if layer_shape is not None:
            self.update_layer_shapes(layer_shape)
        self.precompute_caches()

    def update_layer_shapes(self, layer_shape: Tuple[int, int]) -> None:
        self.layer_shape = layer_shape
        self.layer_shapes = self._compute_downsampled_shapes(self.layer_shape)

    def precompute_caches(self) -> None:
        sizes = tables.block_sizes(self.settings.block_size_range)
        if not hasattr(self, "zigzag_cache"):
            self.zigzag_cache = {}
        for s in sizes:
            if s not in self.zigzag_cache:
                self.zigzag_cache[s] = tables.zigzag_ordering(s)
        self.quantization_matrix_cache = tables.quantization_cache(self.settings.quality_range, self.settings.block_size_range)

    def _compute_downsampled_shapes(self, layer_shapes) -> np.ndarray:
        return np.asarray(layer_shapes) // self.settings.downsampling_ratios          # jpeg.py:676-686

    def _get_quality_factor(self, block_size: int) -> int:
        return tables.quality_factor(block_size, self.settings.quality_range, self.settings.block_size_range)

    @staticmethod
    def _get_quantization_matrix(default_matrix: np.ndarray, size: int, quality: int) -> np.ndarray:
        return tables.quantization_matrix(default_matrix, size, quality)

    @staticmethod
    def _zigzag_ordering(size: int) -> np.ndarray:
        return tables.zigzag_ordering(size)

    # -- public API -----------------------------------------------------------------------------
    def compress(self, img: Image) -> bytes:
        """Compress one image to the .ajpg byte stream (jpeg.py:240-272)."""
        if not isinstance(img, Image):
            raise TypeError("Input must be an Image object.")
        if img.ndim != 3:
            raise ValueError("Input array must be a 3D.")
        return self.compress_batch([img])[0]

    def decompress(self, img_encoded: bytes, scale: int = 1) -> Image:
        """Decode an .ajpg stream (jpeg.py:274-297); reconfigures itself from the stream header.
        scale: 2, 4 or 8 decode a (ceil(H/scale), ceil(W/scale), 3) image straight from the coefficients (previews,
        thumbnails; include/aeaj.h, aeaj_decode_scaled); layer_shape stays the file's full size."""
        return self.decompress_batch([img_encoded], scale=scale)[0]

    def compress_batch(self, imgs: Sequence[Image]) -> List[bytes]:
        """Same-shape images are encoded in one device batch; others fall back to one batch each."""
        for im in imgs:
            if not isinstance(im, Image):
                raise TypeError("Input must be an Image object.")
            if im.ndim != 3:
                raise ValueError("Input array must be a 3D.")
        out: List[Optional[bytes]] = [None] * len(imgs)
        groups = {}
        for i, im in enumerate(imgs):
            groups.setdefault(tuple(im.original_shape[:2]), []).append(i)
        s = self.settings
        codec = get_codec()
        for (H, W), idxs in groups.items():
            self.update_layer_shapes((H, W))
            self.extension = imgs[idxs[-1]].extension
            if all(imgs[i].uint8_source() is not None for i in idxs):
                # 8-bit sources: upload the bytes, the device does astype(float32) / 255.0 (image.py:84)
                host = np.stack([imgs[i].uint8_source().reshape(H, W, 3) for i in idxs])
            else:
                host = np.stack([np.ascontiguousarray(imgs[i].data.reshape(H, W, 3), dtype=np.float32) for i in idxs])
            rgb = torch.from_numpy(host).pin_memory().to(f"cuda:{codec.device}", non_blocking=True)
            enc = codec.encode(rgb, s.color_space, s.quality_range, s.block_size_range, stream=True)
            if self.deflate == "device":
                df = codec.deflate(enc, s.color_space, s.quality_range, s.block_size_range)
                downloaded = codec.download_deflated(enc, df)
                for k, i in enumerate(idxs):
                    out[i] = self._entropy_encode(downloaded[k], (H, W), imgs[i].extension, [L["zlib"] for L in downloaded[k]])
                continue
            downloaded = codec.download(enc)
            # zlib level 9 is the end-to-end bottleneck once the hot path is on the GPU (SURVEY 8f-2): deflate every layer of
            # every image of the group concurrently (zlib releases the GIL; same bytes as the sequential reference loop)
            jobs = [(i, l) for i in range(len(idxs)) for l in range(len(downloaded[i]))]
            with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as pool:
                deflated = list(pool.map(lambda il: self._deflate_layer(downloaded[il[0]][il[1]]), jobs))
            for k, i in enumerate(idxs):
                streams = [deflated[j] for j, (ii, _) in enumerate(jobs) if ii == k]
                out[i] = self._entropy_encode(downloaded[k], (H, W), imgs[i].extension, streams)
        return out

    def decompress_uint8(self, img_encoded: bytes, scale: int = 1) -> np.ndarray:
        """decompress(...).get_uint8() with the (data * 255).astype(uint8) step (image.py:127) done by the decoding
        kernel: a quarter of the device-to-host bytes when only 8-bit pixels are wanted (Image.save, previews)."""
        return self.decompress_batch([img_encoded], as_uint8=True, scale=scale)[0]

    def decompress_batch(self, streams: Sequence[bytes], as_uint8: bool = False, scale: int = 1) -> List[Image]:
        if scale not in (1, 2, 4, 8):
            raise ValueError("scale must be 1, 2, 4 or 8")
        device = self.deflate == "device"
        parsed = [self._entropy_decode(b, inflate=not device) for b in streams]
        out: List[Optional[Image]] = [None] * len(streams)
        groups = {}
        for i, p in enumerate(parsed):
            groups.setdefault((p["H"], p["W"], p["space"], p["quality"], p["blocks"]), []).append(i)
        codec = get_codec()
        for (H, W, space, q, b), idxs in groups.items():
            layers = [parsed[i]["layers"] for i in idxs]
            if device:
                zbuf, offs, lens, leaves, counts = codec.upload_for_inflate(layers, len(idxs), H, W, space, q, b)
                inf = codec.inflate(zbuf, offs, lens, counts, len(idxs), H, W, space, q, b)
                coef = inf.coef
            else:
                coef, leaves, counts = codec.upload_for_decode(layers, len(idxs), H, W, space, q, b)
            rgb = codec.decode(coef, leaves, counts, len(idxs), H, W, space, q, b, zigzag=True, out="u8" if as_uint8 else "f32",
                               scale=scale).cpu().numpy()
            if device:
                _raise_inflate_status(inf.status.cpu().numpy())
            codec.check_status(codec.last_decode_status, "decode")
            for k, i in enumerate(idxs):
                out[i] = rgb[k] if as_uint8 else Image.from_array(rgb[k].reshape(-1, 3), rgb.shape[1:], parsed[i]["extension"])
        last = parsed[-1]
        self.extension = last["extension"]
        self.update_settings(JpegCompressionSettings(last["space"], last["quality"], last["blocks"]), (last["H"], last["W"]))
        return out

    # -- host-side entropy coding (byte-compatible with jpeg.py:531-674) -------------------------
    def _deflate_layer(self, L) -> bytes:
        # With the device-side stream layout the coefficients already arrive zigzag-ordered (jpeg.py:579-590).
        zz = L["coef"] if L.get("zigzag") else _zigzag_stream(L["coef"], L["leaves"][:, 2], self.zigzag_cache, inverse=False)
        return zlib.compress(zz.tobytes(), level=9)

    def _entropy_encode(self, layers, layer_shape, extension, streams=None) -> bytes:
        s = self.settings
        out = BytesIO()
        meta = {"height": int(layer_shape[0]), "width": int(layer_shape[1]), "num_layers": len(layers),
                "color_space": s.color_space, "quality_min": s.quality_range[0], "quality_max": s.quality_range[1],
                "block_size_min": s.block_size_range[0], "block_size_max": s.block_size_range[1], "extension": extension}
        mb = json.dumps(meta).encode("utf-8")
        out.write(len(mb).to_bytes(4, byteorder="big"))
        out.write(mb)
        lib = native.load()

        if streams is None:
            with ThreadPoolExecutor(max_workers=len(layers)) as pool:
                streams = list(pool.map(self._deflate_layer, layers))
        for L, z in zip(layers, streams):
            if "packed_states" in L:
                packed = L["packed_states"]
                n_states = L["n_states"] if "n_states" in L else len(L["states"])
            else:
                states = np.ascontiguousarray(L["states"], dtype=np.uint8)
                n_states = len(states)
                packed = np.empty((len(states) + 3) // 4, dtype=np.uint8)
                native.check(lib.aeaj_pack_states_host(states.ctypes.data, len(states), packed.ctypes.data), "aeaj_pack_states_host")
            out.write((2 * n_states).to_bytes(4, byteorder="big"))
            out.write(int(L["root"]).to_bytes(4, byteorder="big"))
            out.write(packed.tobytes())
            out.write(len(z).to_bytes(4, byteorder="big"))
            out.write(z)
        return out.getvalue()

    def _entropy_decode(self, encoded_data: bytes, inflate: bool = True) -> dict:
        """the .ajpg framing; inflate=False leaves each layer's zlib bytes for the device (zlib, ncoef instead of coef)"""
        s = BytesIO(encoded_data)
        ml = int.from_bytes(s.read(4), byteorder="big")
        meta = json.loads(s.read(ml).decode("utf-8"))
        H, W = meta["height"], meta["width"]
        space = meta["color_space"]
        quality = (meta["quality_min"], meta["quality_max"])
        blocks = (meta["block_size_min"], meta["block_size_max"])
        settings = JpegCompressionSettings(space, quality, blocks)          # raises ValueError on unknown space
        shapes = np.asarray((H, W)) // settings.downsampling_ratios
        layers = []
        for i in range(meta["num_layers"]):
            nbits = int.from_bytes(s.read(4), byteorder="big")
            root = int.from_bytes(s.read(4), byteorder="big")
            raw = np.frombuffer(s.read((nbits + 7) // 8), dtype=np.uint8)
            states = np.stack([(raw >> 6) & 3, (raw >> 4) & 3, (raw >> 2) & 3, raw & 3], axis=1).reshape(-1)[: nbits // 2]
            leaves, ncoef = native.states_to_leaves(states.astype(np.uint8), root, int(shapes[i][0]), int(shapes[i][1]), blocks)
            zl = int.from_bytes(s.read(4), byteorder="big")
            if not inflate:
                layers.append(dict(leaves=leaves, zlib=s.read(zl), ncoef=int(ncoef)))
                continue
            coef = np.frombuffer(zlib.decompress(s.read(zl)), dtype=np.int32)
            if coef.size != ncoef:
                raise ValueError("coefficient stream length does not match the quadtree header")
            layers.append(dict(leaves=leaves, coef=coef))          # still zigzag-ordered: the IDCT kernels undo it on load
        return dict(H=H, W=W, space=space, quality=quality, blocks=blocks, extension=meta["extension"], layers=layers)
