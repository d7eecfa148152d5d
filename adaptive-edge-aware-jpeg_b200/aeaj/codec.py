"""Device pipelines: torch owns device memory and streams, libaeaj.so does the work.

``DeviceCodec`` caches one plan (geometry + q tables + workspace + output buffers) per
(batch, H, W, colour space, block range) and exposes

    encode(rgb_dev)  -> EncodedBatch      Jpeg.compress  minus _entropy_encode (jpeg.py:262-270)
    decode(encoded)  -> rgb_dev           Jpeg.decompress minus _entropy_decode (jpeg.py:285-297)

plus host-buffer variants used by the reference-facing ``Jpeg`` shim and by ``bench.py``'s e2e leg.
Everything is asynchronous on the current torch CUDA stream; nothing falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C
import time
from collections import OrderedDict
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import native, tables


def _require_cuda():
    if not torch.cuda.is_available():
        raise native.AeajError("no CUDA device: the adaptive edge-aware JPEG B200 path has no CPU fallback")


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


@dataclass
class EncodedBatch:
    """Device-resident result of one encode call (buffers are owned by the plan and reused)."""
    coef: List[torch.Tensor]       # 3 x int32 [B, cap_coef_l]
    leaves: List[torch.Tensor]     # 3 x int32 [B, cap_leaves_l, 4]  (x, y, size, coef offset)
    states: List[torch.Tensor]     # 3 x uint8 [B, cap_states_l]
    counts: torch.Tensor           # int32 [B, 3, 4]  n_leaves, n_states, n_coef, root
    status: torch.Tensor           # int32 [64]       [0] hysteresis re-visits, [1] converged, [2] tensor-DCT timeout flag
    shape: Tuple[int, int, int]    # B, H, W
    layers: Optional[List[torch.Tensor]] = None   # taps (float32 [B,h,w]) if requested
    edges: Optional[List[torch.Tensor]] = None    # taps (uint8  [B,h,w]) if requested
    packed_states: Optional[List[torch.Tensor]] = None   # 3 x uint8 [B, (cap_states_l+3)//4] when stream=True
    zigzag: bool = False                          # coefficient blocks are zigzag-ordered (the .ajpg layout)


@dataclass
class PackedBatch:
    """Packed coefficient streams of one batch (include/aeaj.h, aeaj_pack_coefficients): per plane a non-zero bit mask and the
    non-zero values as int16 -- what travels over PCIe to the host-side entropy coder instead of the int32 streams."""
    mask: List[torch.Tensor]       # 3 x int32 [B, cap_coef_l // 32 + 1]   (uint32 words)
    vals: List[torch.Tensor]       # 3 x int16 [B, cap_coef_l]
    counts: torch.Tensor           # int32 [B, 3, 4]  nnz, n_coef, overflow flag, mask words


@dataclass
class DeflatedBatch:
    """Device deflate of one batch's coefficient streams (include/aeaj.h, aeaj_deflate_coefficients): per plane one complete
    zlib stream, readable by any inflate -- what travels over PCIe to the .ajpg writer instead of the int32 streams."""
    out: List[torch.Tensor]        # 3 x uint8 [B, cap_out_l]
    lengths: torch.Tensor          # int32 [B, 3]  bytes of each stream
    status: torch.Tensor           # int32 [4]     [0] planes whose stream did not fit (0 = ok)


@dataclass
class InflatedBatch:
    """Device inflate of one batch's zlib streams into the plan's coefficient buffers (include/aeaj.h,
    aeaj_inflate_coefficients); the per-plane results stay on the device until read."""
    coef: List[torch.Tensor]       # 3 x int32 [B, cap_coef_l]: the plan's buffers, as aeaj_decode reads them
    status: torch.Tensor           # int32 [B, 3]  0 ok, else the INFLATE_ERRORS code
    out_bytes: torch.Tensor        # int64 [B, 3]  bytes written
    segments: torch.Tensor         # int32 [B, 3]  parts decoded independently (sync points of the stream)


# statuses of aeaj_inflate_coefficients (csrc/inflate_core.h), worded like zlib's messages
INFLATE_ERRORS = {1: "incorrect header check", 2: "preset dictionary required", 3: "invalid block type",
                  4: "invalid stored block lengths", 5: "invalid code lengths", 6: "invalid literal/length or distance code",
                  7: "invalid distance too far back", 8: "incomplete or truncated stream", 9: "incorrect data check",
                  10: "coefficient stream length does not match the quadtree header"}
INFLATE_LENGTH = 10


@dataclass
class _HostStaging:
    """Buffers of one stream slot of roundtrip_host_pipelined (one frame per job): pinned host memory for what crosses PCIe
    in per-range copies, and the device-side input frame and arena."""
    coef: List[torch.Tensor]       # 3 x int32 [cap_coef_l]     pinned
    leaves: List[torch.Tensor]     # 3 x int32 [cap_leaves_l, 4]
    states: List[torch.Tensor]     # 3 x uint8 [cap_states_l]
    counts: torch.Tensor           # int32 [1, 3, 4]  of EncodedBatch.counts
    pk_counts: torch.Tensor        # int32 [1, 3, 4]  of PackedBatch.counts
    rgb_dev: Dict[torch.dtype, torch.Tensor] = field(default_factory=dict)   # device input frame [1,H,W,3] per pixel dtype used
    arena_dev: Optional[torch.Tensor] = None       # a frame's packed streams, contiguous (device and pinned host)
    arena_host: Optional[torch.Tensor] = None


@dataclass
class _Job:
    """One frame in flight in roundtrip_host_pipelined."""
    frame: int                     # index into host_in / host_out
    slot: int                      # stream and plan instance
    p: _Plan
    enc: EncodedBatch
    encoded: torch.cuda.Event      # phase A done: the counts are on the host
    decoded: Optional[torch.cuda.Event] = None    # recorded after the job's last copy, when phase B is issued


@dataclass
class _Scaled:
    """A plan's buffers for decode(..., scale=k), k > 1 (aeaj_decode_scaled)."""
    out_h: int
    out_w: int
    layer_h: Tuple[int, int, int]  # the final scaled layers
    layer_w: Tuple[int, int, int]
    scratch: torch.Tensor          # the scaled layers of the call
    rgb_out: torch.Tensor          # float32 [B, out_h, out_w, 3]
    rgb8_out: Optional[torch.Tensor] = None


@dataclass
class _Plan:
    ptr: C.c_void_p
    info: native.PlanInfo
    workspace: torch.Tensor
    out: EncodedBatch
    rgb_out: torch.Tensor
    rgb8_out: Optional[torch.Tensor] = None
    qkey: Optional[tuple] = None
    staging: Optional[_HostStaging] = None
    dec_status: Optional[torch.Tensor] = None     # int32 [64]: [2] tensor-IDCT timeout flag, [3] leaves rejected by the device guard
    packed: Optional[PackedBatch] = None
    deflated: Optional[DeflatedBatch] = None
    deflate_scratch: Optional[torch.Tensor] = None
    inflated: Optional[InflatedBatch] = None
    inflate_scratch: Optional[torch.Tensor] = None
    scaled: Dict[int, _Scaled] = field(default_factory=dict)
    nbytes: int = 0


class DeviceCodec:
    MAX_PLANS = 48                      # plans (geometry + workspace + output buffers) kept per device, least recently used first out
    MAX_PLAN_BYTES = 96 << 30           # ... and the device memory they may hold together

    def __init__(self, device: int = 0):
        _require_cuda()
        self.device = device
        self.lib = native.load()
        self.handle = native.handle(device)
        self._plans: "OrderedDict[tuple, _Plan]" = OrderedDict()
        self.last_launches = 0
        # size classes whose DCT / IDCT run on the tcgen05 / TMEM kernels: bit k = class 16 << k (True = all four, False / 0 =
        # the FP32-FMA kernels everywhere).  Default: 32 x 32 and 128 x 128 -- measured on B200 (profiles/r2_tc_variants.md) the
        # FP32 kernels are as fast for 64 and faster for 16
        self.tensor_dct = 0xa

    def _tensor_mask(self) -> int:
        return 0xf if self.tensor_dct is True else int(self.tensor_dct) & 0xf

    def tensor_dct_timed_out(self) -> bool:
        t = (C.c_int * 32)()
        native.check(self.lib.aeaj_tensor_dct_status(self.handle, C.cast(t, C.POINTER(C.c_int))), "aeaj_tensor_dct_status")
        self.tensor_dct_phase_cycles = list(t)[1:16]
        return bool(t[0])

    # ------------------------------------------------------------------------------------------
    def _plan(self, B, H, W, space, brange, qrange, instance: int = 0) -> _Plan:
        key = (B, H, W, space, tuple(brange), instance)
        p = self._plans.get(key)
        dev = torch.device("cuda", self.device)
        if p is not None:
            self._plans.move_to_end(key)
        if p is None:
            if space not in tables.CODEC_SPACES:
                raise ValueError(f"Unsupported color space: {space}")
            ptr = C.c_void_p()
            native.check(self.lib.aeaj_plan_create(self.handle, B, H, W, tables.SPACE_ID[space], brange[0], brange[1], C.byref(ptr)),
                         "aeaj_plan_create")
            info = native.PlanInfo()
            native.check(self.lib.aeaj_plan_get_info(ptr, C.byref(info)), "aeaj_plan_get_info")
            ws = torch.empty(int(info.workspace_bytes), dtype=torch.uint8, device=dev)
            out = EncodedBatch(
                coef=[torch.empty((B, int(info.cap_coef[l])), dtype=torch.int32, device=dev) for l in range(3)],
                leaves=[torch.empty((B, int(info.cap_leaves[l]), 4), dtype=torch.int32, device=dev) for l in range(3)],
                states=[torch.empty((B, int(info.cap_states[l])), dtype=torch.uint8, device=dev) for l in range(3)],
                counts=torch.zeros((B, 3, 4), dtype=torch.int32, device=dev),
                status=torch.zeros(64, dtype=torch.int32, device=dev), shape=(B, H, W))
            rgb_out = torch.empty((B, H, W, 3), dtype=torch.float32, device=dev)
            p = _Plan(ptr, info, ws, out, rgb_out, dec_status=torch.zeros(64, dtype=torch.int32, device=dev))
            p.nbytes = ws.numel() + rgb_out.numel() * 4 + sum(t.numel() * t.element_size() for t in out.coef + out.leaves + out.states)
            self._plans[key] = p
            self._evict(keep=key)
        qkey = tuple(qrange)
        if p.qkey != qkey:
            cache = tables.quantization_cache(qrange, brange)
            sizes = tables.block_sizes(brange)
            flat = np.concatenate([cache[t][s].ravel() for t in (0, 1) for s in sizes]).astype(np.int32)
            native.check(self.lib.aeaj_plan_set_qtables(p.ptr, flat.ctypes.data, flat.size, _stream()), "aeaj_plan_set_qtables")
            torch.cuda.current_stream().synchronize()     # `flat` is pageable host memory
            p.qkey = qkey
        return p

    def _evict(self, keep=None):
        """Bound the plan cache (a dataset of mixed image sizes would otherwise hold a workspace per distinct shape until OOM)."""
        def total():
            return sum(q.nbytes for q in self._plans.values())
        while len(self._plans) > 1 and (len(self._plans) > self.MAX_PLANS or total() > self.MAX_PLAN_BYTES):
            key = next(k for k in self._plans if k != keep)
            old = self._plans.pop(key)
            torch.cuda.synchronize(self.device)          # nothing in flight may still read the plan's device tables
            native.check(self.lib.aeaj_plan_destroy(old.ptr), "aeaj_plan_destroy")
            old.ptr = None

    def close(self):
        """Destroy every cached plan (their tensors are freed by torch once unreferenced)."""
        torch.cuda.synchronize(self.device)
        while self._plans:
            _, old = self._plans.popitem(last=False)
            native.check(self.lib.aeaj_plan_destroy(old.ptr), "aeaj_plan_destroy")
            old.ptr = None

    def check_status(self, status: torch.Tensor, what: str = "encode"):
        """Raise if the device reported a problem for the call that wrote `status` (synchronises the stream)."""
        s = status[:4].cpu().numpy()
        if what == "encode" and int(s[1]) != 1:
            raise native.AeajError("hysteresis did not converge")
        if int(s[2]) == 2:
            raise native.AeajError("a rank did not reach a peer barrier of the multi-GPU halo-split within its time limit; the results are invalid")
        if int(s[2]) != 0:
            raise native.AeajError("the tensor-core DCT kernel timed out on a barrier wait; its coefficients are invalid")
        if what == "decode" and int(s[3]) != 0:
            raise ValueError(f"{int(s[3])} leaves do not fit the layer geometry / block range (corrupt stream)")

    def plan_info(self, B, H, W, space, brange, qrange=(40, 80)) -> native.PlanInfo:
        return self._plan(B, H, W, space, brange, qrange).info

    # ------------------------------------------------------------------------------------------
    def encode(self, rgb: torch.Tensor, space: str, qrange, brange, taps: bool = False, instance: int = 0,
               stream: bool = False) -> EncodedBatch:
        """rgb: float32 CUDA tensor [B,H,W,3] (or [H,W,3]) in [0,1] -- or uint8 pixels, converted on the device exactly
        as Image.load does (astype(float32) / 255.0, image.py:84).  Asynchronous on the current stream.
        stream=True produces the .ajpg stream layout on the device: zigzag-ordered coefficient blocks and the
        2-bit packed state stream (what _entropy_encode feeds to zlib / writes, jpeg.py:563-590)."""
        if rgb.dim() == 3:
            rgb = rgb.unsqueeze(0)
        if rgb.dtype not in (torch.float32, torch.uint8) or not rgb.is_cuda or rgb.dim() != 4 or rgb.shape[-1] != 3:
            raise TypeError("encode expects a float32 (or uint8) CUDA tensor of shape [B,H,W,3]")
        rgb = rgb.contiguous()
        B, H, W, _ = rgb.shape
        p = self._plan(B, H, W, space, brange, qrange, instance)
        o = p.out
        io = native.EncodeIO()
        if rgb.dtype == torch.uint8:
            io.rgb_u8 = rgb.data_ptr()
        else:
            io.rgb = rgb.data_ptr()
        for l in range(3):
            io.coef[l] = o.coef[l].data_ptr()
            io.leaves[l] = o.leaves[l].data_ptr()
            io.states[l] = o.states[l].data_ptr()
        io.counts = o.counts.data_ptr()
        io.status = o.status.data_ptr()
        native.check(self.lib.aeaj_plan_set_stream_layout(p.ptr, int(stream)), "aeaj_plan_set_stream_layout")
        native.check(self.lib.aeaj_plan_set_tensor_dct(p.ptr, self._tensor_mask()), "aeaj_plan_set_tensor_dct")
        o.zigzag = bool(stream)
        if stream:
            if o.packed_states is None:
                o.packed_states = [torch.empty((B, (int(p.info.cap_states[l]) + 3) // 4), dtype=torch.uint8, device=rgb.device) for l in range(3)]
            for l in range(3):
                io.packed_states[l] = o.packed_states[l].data_ptr()
        if taps:
            dev = rgb.device
            o.layers = [torch.empty((B, p.info.layer_h[l], p.info.layer_w[l]), dtype=torch.float32, device=dev) for l in range(3)]
            o.edges = [torch.empty((B, p.info.layer_h[l], p.info.layer_w[l]), dtype=torch.uint8, device=dev) for l in range(3)]
            for l in range(3):
                io.tap_layers[l] = o.layers[l].data_ptr()
                io.tap_edges[l] = o.edges[l].data_ptr()
        native.check(self.lib.aeaj_encode(p.ptr, C.byref(io), p.workspace.data_ptr(), _stream()), "aeaj_encode")
        self.last_launches = self.lib.aeaj_plan_last_launches(p.ptr)
        return o

    def decode(self, coef, leaves, counts, B, H, W, space: str, qrange, brange, taps: bool = False, instance: int = 0,
               zigzag: bool = False, out: str = "f32", scale: int = 1):
        """coef/leaves: 3 device tensors laid out like EncodedBatch; counts int32 [B,3,4]. Returns rgb [B,H,W,3].
        zigzag=True: the coefficient blocks are in the .ajpg zigzag order.
        out: "f32" (Image.data), "u8" (Image.get_uint8(), (data * 255).astype(uint8), written by the same kernel) or "both"
        (returns the pair).
        scale: 2, 4 or 8 decode at 1/scale of the size, straight from the coefficients (aeaj_decode_scaled, include/aeaj.h) and
        return rgb [B, ceil(H/scale), ceil(W/scale), 3] (taps: the scaled layers); 1 is the full-size decode."""
        if out not in ("f32", "u8", "both"):
            raise ValueError("out must be 'f32', 'u8' or 'both'")
        if scale not in (1, 2, 4, 8):
            raise ValueError("scale must be 1, 2, 4 or 8")
        p = self._plan(B, H, W, space, brange, qrange, instance)
        if scale != 1:
            return self._decode_scaled(p, coef, leaves, counts, B, taps, zigzag, out, scale)
        native.check(self.lib.aeaj_plan_set_stream_layout(p.ptr, int(zigzag)), "aeaj_plan_set_stream_layout")
        native.check(self.lib.aeaj_plan_set_tensor_dct(p.ptr, self._tensor_mask()), "aeaj_plan_set_tensor_dct")
        io = native.DecodeIO()
        for l in range(3):
            if coef[l].shape[1] != p.info.cap_coef[l] or leaves[l].shape[1] != p.info.cap_leaves[l]:
                raise ValueError("decode buffers must use the plan's capacities")
            io.coef[l] = coef[l].data_ptr()
            io.leaves[l] = leaves[l].data_ptr()
        io.counts = counts.data_ptr()
        if out != "u8":
            io.rgb = p.rgb_out.data_ptr()
        if out != "f32":
            if p.rgb8_out is None:
                p.rgb8_out = torch.empty((B, H, W, 3), dtype=torch.uint8, device=p.rgb_out.device)
            io.rgb_u8 = p.rgb8_out.data_ptr()
        io.status = p.dec_status.data_ptr()
        self.last_decode_status = p.dec_status
        tl = None
        if taps:
            tl = [torch.empty((B, p.info.layer_h[l], p.info.layer_w[l]), dtype=torch.float32, device=p.rgb_out.device) for l in range(3)]
            for l in range(3):
                io.tap_layers[l] = tl[l].data_ptr()
        native.check(self.lib.aeaj_decode(p.ptr, C.byref(io), p.workspace.data_ptr(), _stream()), "aeaj_decode")
        self.last_launches = self.lib.aeaj_plan_last_launches(p.ptr)
        res = p.rgb_out if out == "f32" else (p.rgb8_out if out == "u8" else (p.rgb_out, p.rgb8_out))
        return (res, tl) if taps else res

    def _scaled(self, p: _Plan, scale: int) -> _Scaled:
        sc = p.scaled.get(scale)
        if sc is None:
            oh, ow, scratch = C.c_int(), C.c_int(), C.c_int64()
            lh, lw = (C.c_int * 3)(), (C.c_int * 3)()
            native.check(self.lib.aeaj_decode_scaled_geometry(p.ptr, scale, C.byref(oh), C.byref(ow), lh, lw, C.byref(scratch)),
                         "aeaj_decode_scaled_geometry")
            dev = p.rgb_out.device
            sc = _Scaled(oh.value, ow.value, tuple(lh), tuple(lw), torch.empty(int(scratch.value), dtype=torch.uint8, device=dev),
                         torch.empty((p.info.batch, oh.value, ow.value, 3), dtype=torch.float32, device=dev))
            p.scaled[scale] = sc
            p.nbytes += sc.scratch.numel() + sc.rgb_out.numel() * 4
            self._evict(keep=next(k for k, v in self._plans.items() if v is p))
        return sc

    def _decode_scaled(self, p: _Plan, coef, leaves, counts, B, taps, zigzag, out, scale):
        sc = self._scaled(p, scale)
        native.check(self.lib.aeaj_plan_set_stream_layout(p.ptr, int(zigzag)), "aeaj_plan_set_stream_layout")
        io = native.DecodeIO()
        for l in range(3):
            if coef[l].shape[1] != p.info.cap_coef[l] or leaves[l].shape[1] != p.info.cap_leaves[l]:
                raise ValueError("decode buffers must use the plan's capacities")
            io.coef[l] = coef[l].data_ptr()
            io.leaves[l] = leaves[l].data_ptr()
        io.counts = counts.data_ptr()
        if out != "u8":
            io.rgb = sc.rgb_out.data_ptr()
        if out != "f32":
            if sc.rgb8_out is None:
                sc.rgb8_out = torch.empty(sc.rgb_out.shape, dtype=torch.uint8, device=sc.rgb_out.device)
                p.nbytes += sc.rgb8_out.numel()
            io.rgb_u8 = sc.rgb8_out.data_ptr()
        io.status = p.dec_status.data_ptr()
        self.last_decode_status = p.dec_status
        tl = None
        if taps:
            tl = [torch.empty((B, sc.layer_h[l], sc.layer_w[l]), dtype=torch.float32, device=sc.rgb_out.device) for l in range(3)]
            for l in range(3):
                io.tap_layers[l] = tl[l].data_ptr()
        native.check(self.lib.aeaj_decode_scaled(p.ptr, C.byref(io), scale, p.workspace.data_ptr(), sc.scratch.data_ptr(), _stream()),
                     "aeaj_decode_scaled")
        self.last_launches = self.lib.aeaj_plan_last_launches(p.ptr)
        res = sc.rgb_out if out == "f32" else (sc.rgb8_out if out == "u8" else (sc.rgb_out, sc.rgb8_out))
        return (res, tl) if taps else res

    # ------------------------------------------------------------------------------------------
    # packed coefficient streams (PCIe form)
    # ------------------------------------------------------------------------------------------
    def _packed(self, p: _Plan) -> PackedBatch:
        if p.packed is None:
            B, dev = p.info.batch, p.rgb_out.device
            p.packed = PackedBatch(mask=[torch.empty((B, int(p.info.cap_coef[l]) // 32 + 1), dtype=torch.int32, device=dev) for l in range(3)],
                                   vals=[torch.empty((B, int(p.info.cap_coef[l])), dtype=torch.int16, device=dev) for l in range(3)],
                                   counts=torch.zeros((B, 3, 4), dtype=torch.int32, device=dev))
            p.nbytes += sum(t.numel() * t.element_size() for t in p.packed.mask + p.packed.vals)
        return p.packed

    def pack(self, enc: EncodedBatch, space, qrange, brange, instance: int = 0) -> PackedBatch:
        """Lossless packed form of enc.coef (bit mask + int16 non-zeros) in the plan's packed buffers; asynchronous."""
        B, H, W = enc.shape
        p = self._plan(B, H, W, space, brange, qrange, instance)
        pk = self._packed(p)
        io = native.PackedIO()
        coef = (C.c_void_p * 3)(*[enc.coef[l].data_ptr() for l in range(3)])
        for l in range(3):
            io.mask[l], io.vals[l] = pk.mask[l].data_ptr(), pk.vals[l].data_ptr()
        io.counts = pk.counts.data_ptr()
        native.check(self.lib.aeaj_pack_coefficients(p.ptr, coef, enc.counts.data_ptr(), C.byref(io), p.workspace.data_ptr(), _stream()),
                     "aeaj_pack_coefficients")
        return pk

    def _deflated(self, p: _Plan) -> DeflatedBatch:
        if p.deflated is None:
            B, dev = p.info.batch, p.rgb_out.device
            cap = (C.c_int64 * 3)()
            scratch = C.c_int64()
            native.check(self.lib.aeaj_deflate_caps(p.ptr, cap, C.byref(scratch)), "aeaj_deflate_caps")
            p.deflated = DeflatedBatch(out=[torch.empty((B, int(cap[l])), dtype=torch.uint8, device=dev) for l in range(3)],
                                       lengths=torch.zeros((B, 3), dtype=torch.int32, device=dev),
                                       status=torch.zeros(4, dtype=torch.int32, device=dev))
            p.deflate_scratch = torch.empty(int(scratch.value), dtype=torch.uint8, device=dev)
            p.nbytes += sum(t.numel() for t in p.deflated.out) + p.deflate_scratch.numel()
            self._evict(keep=next(k for k, v in self._plans.items() if v is p))
        return p.deflated

    def deflate(self, enc: EncodedBatch, space, qrange, brange, instance: int = 0) -> DeflatedBatch:
        """One zlib stream per plane of enc.coef, on the device (aeaj_deflate_coefficients): the entropy coder of the .ajpg
        container without the int32 streams crossing PCIe.  With encode(stream=True) the payloads are exactly the streams the
        host path hands to zlib.  Asynchronous; the buffers belong to the plan and are reused by the next call."""
        B, H, W = enc.shape
        p = self._plan(B, H, W, space, brange, qrange, instance)
        df = self._deflated(p)
        io = native.DeflateIO()
        for l in range(3):
            io.out[l] = df.out[l].data_ptr()
        io.lengths = df.lengths.data_ptr()
        io.status = df.status.data_ptr()
        coef = (C.c_void_p * 3)(*[enc.coef[l].data_ptr() for l in range(3)])
        native.check(self.lib.aeaj_deflate_coefficients(p.ptr, coef, enc.counts.data_ptr(), C.byref(io), p.deflate_scratch.data_ptr(),
                                                         _stream()), "aeaj_deflate_coefficients")
        return df

    def download_deflated(self, enc: EncodedBatch, df: DeflatedBatch):
        """D2H of what the .ajpg writer needs after deflate() of an encode(stream=True) batch: per image a list of 3
        dicts(zlib, packed_states, n_states, root) -- the used zlib bytes, the packed state streams and the counts; the
        coefficients stay on the device.  Synchronises the stream."""
        if not enc.zigzag or enc.packed_states is None:
            raise ValueError("download_deflated needs the .ajpg stream layout: encode(..., stream=True)")
        counts = enc.counts.cpu().numpy()
        lengths = df.lengths.cpu().numpy()
        self.check_status(enc.status, "encode")
        if int(df.status[0].item()) != 0:
            raise native.AeajError("a deflated coefficient stream did not fit its buffer")
        out = []
        for b in range(enc.shape[0]):
            layers = []
            for l in range(3):
                ns, root = int(counts[b, l, 1]), int(counts[b, l, 3])
                layers.append(dict(zlib=df.out[l][b, :int(lengths[b, l])].cpu().numpy().tobytes(),
                                   packed_states=enc.packed_states[l][b, :(ns + 3) // 4].cpu().numpy(), n_states=ns, root=root))
            out.append(layers)
        return out

    def inflate(self, zbuf: torch.Tensor, offsets: torch.Tensor, lengths: torch.Tensor, counts: torch.Tensor, B, H, W, space,
                qrange, brange, instance: int = 0) -> InflatedBatch:
        """Inflate plane (b, l)'s zlib stream zbuf[offsets[b, l] : + lengths[b, l]] (device uint8; int64 [B, 3] device
        arrays) into the plan's coefficient buffers, on the device (aeaj_inflate_coefficients): the .ajpg reader's zlib
        layer without the int32 streams crossing PCIe.  Each stream must inflate to exactly 4 * counts[b, l, 2] bytes
        (counts as decode() takes them).  Asynchronous; the results belong to the plan and are reused by the next call."""
        p = self._plan(B, H, W, space, brange, qrange, instance)
        if zbuf.dtype != torch.uint8 or not zbuf.is_cuda or not zbuf.is_contiguous():
            raise TypeError("inflate expects a contiguous uint8 CUDA tensor")
        for t, dt in ((offsets, torch.int64), (lengths, torch.int64), (counts, torch.int32)):
            if t.dtype != dt or not t.is_cuda or not t.is_contiguous() or t.shape[:2] != (B, 3):
                raise TypeError("offsets / lengths: int64 [B, 3], counts: int32 [B, 3, 4], contiguous CUDA tensors")
        dev = p.rgb_out.device
        if p.inflated is None:
            p.inflated = InflatedBatch(coef=p.out.coef, status=torch.zeros((B, 3), dtype=torch.int32, device=dev),
                                       out_bytes=torch.zeros((B, 3), dtype=torch.int64, device=dev),
                                       segments=torch.zeros((B, 3), dtype=torch.int32, device=dev))
        need = C.c_int64()
        native.check(self.lib.aeaj_inflate_scratch_bytes(p.ptr, zbuf.numel(), C.byref(need)), "aeaj_inflate_scratch_bytes")
        if p.inflate_scratch is None or p.inflate_scratch.numel() < need.value:
            if p.inflate_scratch is not None:
                p.nbytes -= p.inflate_scratch.numel()
            p.inflate_scratch = torch.empty(int(need.value), dtype=torch.uint8, device=dev)
            p.nbytes += p.inflate_scratch.numel()
            self._evict(keep=next(k for k, v in self._plans.items() if v is p))
        ib = p.inflated
        io = native.InflateIO()
        io.inp = zbuf.data_ptr() if zbuf.numel() else None
        io.offsets, io.lengths = offsets.data_ptr(), lengths.data_ptr()
        for l in range(3):
            io.coef[l] = ib.coef[l].data_ptr()
        io.status, io.out_bytes, io.segments = ib.status.data_ptr(), ib.out_bytes.data_ptr(), ib.segments.data_ptr()
        native.check(self.lib.aeaj_inflate_coefficients(p.ptr, C.byref(io), counts.data_ptr(), zbuf.numel(),
                                                        p.inflate_scratch.data_ptr(), _stream()), "aeaj_inflate_coefficients")
        return ib

    def upload_for_inflate(self, per_image_layers, B, H, W, space, qrange, brange):
        """per_image_layers[b][l] = dict(leaves (n,4) int32 incl. coef offsets, zlib bytes, ncoef): the zlib bytes, leaves,
        counts, offsets and lengths in ONE pinned host-to-device copy; the leaves land in the plan's buffers.  Returns the
        device (zbuf, offsets, lengths, leaves, counts); asynchronous."""
        p = self._plan(B, H, W, space, brange, qrange)
        o = p.out
        counts = np.zeros((B, 3, 4), dtype=np.int32)
        offs = np.zeros((B, 3), dtype=np.int64)
        lens = np.zeros((B, 3), dtype=np.int64)
        zl = 0
        for b in range(B):
            for l in range(3):
                d = per_image_layers[b][l]
                nl = len(d["leaves"])
                if nl > p.info.cap_leaves[l] or d["ncoef"] > p.info.cap_coef[l]:
                    raise ValueError("stream does not fit the layer geometry (corrupt input?)")
                counts[b, l, 0], counts[b, l, 2] = nl, d["ncoef"]
                offs[b, l], lens[b, l] = zl, len(d["zlib"])
                zl += len(d["zlib"])
        zpad = (zl + 15) & ~15
        nleaf = [[len(per_image_layers[b][l]["leaves"]) * 16 for l in range(3)] for b in range(B)]
        total = zpad + sum(map(sum, nleaf)) + counts.nbytes + offs.nbytes + lens.nbytes
        host = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        h = host.numpy()
        pos = 0
        for b in range(B):
            for l in range(3):
                z = per_image_layers[b][l]["zlib"]
                h[pos:pos + len(z)] = np.frombuffer(z, dtype=np.uint8)
                pos += len(z)
        pos = zpad
        for b in range(B):
            for l in range(3):
                n = nleaf[b][l]
                h[pos:pos + n] = np.require(per_image_layers[b][l]["leaves"], dtype=np.int32, requirements=["C"]).view(np.uint8).ravel()
                pos += n
        tail = pos
        for a in (counts, offs, lens):
            h[pos:pos + a.nbytes] = a.view(np.uint8).ravel()
            pos += a.nbytes
        dev = host.to(p.rgb_out.device, non_blocking=True)
        pos = zpad
        for b in range(B):
            for l in range(3):
                n = nleaf[b][l]
                if n:
                    o.leaves[l][b, :n // 16].view(-1).view(torch.uint8).copy_(dev[pos:pos + n], non_blocking=True)
                pos += n
        o.counts.view(-1).view(torch.uint8).copy_(dev[tail:tail + counts.nbytes], non_blocking=True)
        pos = tail + counts.nbytes
        d_offs = dev[pos:pos + offs.nbytes].view(torch.int64).view(B, 3)
        d_lens = dev[pos + offs.nbytes:pos + offs.nbytes + lens.nbytes].view(torch.int64).view(B, 3)
        return dev[:zl], d_offs, d_lens, o.leaves, o.counts

    def unpack(self, pk: PackedBatch, B, H, W, space, qrange, brange, instance: int = 0) -> List[torch.Tensor]:
        """Inverse of pack(): expands into the plan's int32 coefficient buffers (returned); asynchronous."""
        p = self._plan(B, H, W, space, brange, qrange, instance)
        io = native.PackedIO()
        coef = (C.c_void_p * 3)(*[p.out.coef[l].data_ptr() for l in range(3)])
        for l in range(3):
            io.mask[l], io.vals[l] = pk.mask[l].data_ptr(), pk.vals[l].data_ptr()
        io.counts = pk.counts.data_ptr()
        native.check(self.lib.aeaj_unpack_coefficients(p.ptr, C.byref(io), coef, p.workspace.data_ptr(), _stream()), "aeaj_unpack_coefficients")
        return p.out.coef

    def capture_roundtrip(self, rgb: torch.Tensor, space, qrange, brange, out: str = "f32"):
        """CUDA-graph capture of encode + decode of `rgb` (the per-call launches -- ~25 kernels and a few memsets -- become one
        graph launch; for single-image latency).  Steady-state calls issue no host-to-device copy, so they are capturable after
        one eager warm-up call.  Returns (graph, result tensor); replay with graph.replay()."""
        if rgb.dim() == 3:
            rgb = rgb.unsqueeze(0)
        B, H, W, _ = rgb.shape
        side = torch.cuda.Stream(device=rgb.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):                                     # warm-up on the capture stream: tables, plane descriptors
                enc = self.encode(rgb, space, qrange, brange, instance=2000)
                res = self.decode(enc.coef, enc.leaves, enc.counts, B, H, W, space, qrange, brange, instance=2000, out=out)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize(rgb.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            enc = self.encode(rgb, space, qrange, brange, instance=2000)
            res = self.decode(enc.coef, enc.leaves, enc.counts, B, H, W, space, qrange, brange, instance=2000, out=out)
        return g, res

    def roundtrip_device(self, rgb: torch.Tensor, space: str, qrange, brange, streams: int = 2, out: str = "f32"):
        """encode + decode of a device-resident batch, split into `streams` sub-batches that run concurrently on their
        own CUDA streams (and plan instances): the latency-bound stages of one sub-batch (hysteresis rounds, quadtree
        scans) overlap the throughput-bound stages of the other.  Fork / join around the current stream, so to the
        caller it behaves like one asynchronous call.  Returns the list of per-sub-batch results (views of plan buffers)."""
        B = rgb.shape[0]
        n = max(1, min(streams, B))
        if not hasattr(self, "_rt_streams") or len(self._rt_streams) < n:
            self._rt_streams = [torch.cuda.Stream(device=rgb.device) for _ in range(n)]
        main = torch.cuda.current_stream()
        fork = torch.cuda.Event()
        fork.record(main)
        H, W = rgb.shape[1], rgb.shape[2]
        outs, launches = [], 0
        for i, part in enumerate(rgb.chunk(n)):
            s = self._rt_streams[i]
            s.wait_event(fork)
            with torch.cuda.stream(s):
                enc = self.encode(part, space, qrange, brange, instance=1000 + i)
                launches += self.last_launches
                outs.append(self.decode(enc.coef, enc.leaves, enc.counts, part.shape[0], H, W, space, qrange, brange, instance=1000 + i, out=out))
                launches += self.last_launches
            join = torch.cuda.Event()
            join.record(s)
            main.wait_event(join)
        self.last_launches = launches
        return outs

    # ------------------------------------------------------------------------------------------
    # measurement support
    # ------------------------------------------------------------------------------------------
    def enable_timing(self, B, H, W, space, brange, qrange, on: bool):
        p = self._plan(B, H, W, space, brange, qrange)
        native.check(self.lib.aeaj_plan_enable_timing(p.ptr, int(on)), "aeaj_plan_enable_timing")

    def read_timing(self, B, H, W, space, brange, qrange) -> Dict[str, float]:
        """Stage durations (ms) of the last encode or decode call on this plan (CUDA events)."""
        p = self._plan(B, H, W, space, brange, qrange)
        names = C.create_string_buffer(4096)
        ms = (C.c_float * 64)()
        n = C.c_int()
        native.check(self.lib.aeaj_plan_read_timing(p.ptr, names, 4096, ms, 64, C.byref(n)), "aeaj_plan_read_timing")
        return {nm: float(ms[i]) for i, nm in enumerate(names.value.decode().split("\n")[: n.value])}

    # ------------------------------------------------------------------------------------------
    # host-buffer path (what a caller holding numpy / pinned host memory uses; bench.py e2e leg)
    # ------------------------------------------------------------------------------------------
    def _host_staging(self, p: _Plan) -> _HostStaging:
        if p.staging is None:
            info = p.info
            p.staging = _HostStaging(
                coef=[torch.empty(int(info.cap_coef[l]), dtype=torch.int32).pin_memory() for l in range(3)],
                leaves=[torch.empty((int(info.cap_leaves[l]), 4), dtype=torch.int32).pin_memory() for l in range(3)],
                states=[torch.empty(int(info.cap_states[l]), dtype=torch.uint8).pin_memory() for l in range(3)],
                counts=torch.empty((1, 3, 4), dtype=torch.int32).pin_memory(),
                pk_counts=torch.empty((1, 3, 4), dtype=torch.int32).pin_memory())
        return p.staging

    def _arena(self, p: _Plan):
        """one contiguous device + pinned-host buffer that holds a whole frame's packed streams (mask words, int16 values,
        leaves, states of the three layers), so that a frame travels in ONE copy per direction (aeaj_copy_segments)"""
        st = p.staging
        if st.arena_dev is None:
            n = 0
            for l in range(3):
                cc = int(p.info.cap_coef[l])
                n += (cc // 32 + 1) * 4 + cc * 2 + int(p.info.cap_leaves[l]) * 16 + int(p.info.cap_states[l]) + 4 * 32
            st.arena_dev = torch.empty(n, dtype=torch.uint8, device=p.rgb_out.device)
            st.arena_host = torch.empty(n, dtype=torch.uint8).pin_memory()
        return st.arena_dev, st.arena_host

    def _copy_segments(self, segs):
        """(src, dst, bytes) ranges in one launch; a frame has 12, within the 64 that travel in the kernel parameters"""
        arr = (native.Segment * len(segs))()
        for k, (src, dst, nb) in enumerate(segs):
            arr[k].src, arr[k].dst, arr[k].bytes = src, dst, nb
        native.check(self.lib.aeaj_copy_segments(arr, len(segs), None, _stream()), "aeaj_copy_segments")

    def roundtrip_host_pipelined(self, host_in: torch.Tensor, host_out: torch.Tensor, space, qrange, brange, slots: int = 8, repeat: int = 1,
                                 lag: int = 3, packed: bool = True):
        """Host-buffer encode+decode of every frame of `host_in` (pinned float32 -- or uint8, the 8-bit image flow
        Image.load -> compress ... decompress -> Image.save -- [F,H,W,3]) into `host_out` (float32 or uint8), one frame per
        job, jobs round-robin over `slots` CUDA streams so that the H2D and D2H copies of different jobs overlap each other
        and the kernels (PCIe is full duplex; the step is copy-bound).  Per job, in stream order:
        H2D RGB -> aeaj_encode -> D2H counts -> [host waits for the counts] -> D2H of the job's streams ->
        H2D of the same bytes (what a host-side entropy decoder would hand back) -> aeaj_decode -> D2H RGB.
        The host waits for a job's counts `lag` jobs later (at most slots - 1), so that the wait normally does not block.
        `repeat` > 1 streams the same F frames that many times back to back (a long-running ingest) without draining
        the pipeline in between.  packed=True moves the coefficient streams in their packed form (bit mask + int16 non-zeros,
        aeaj_pack_coefficients after the encode, aeaj_unpack_coefficients before the decode) and all of a job's streams as ONE
        copy per direction (aeaj_copy_segments); a job in which any plane overflows int16 travels as with packed=False:
        raw int32 streams, one copy per range.
        Measured on B200 (tools/e2e_sweep.py, profiles/r2_e2e_sweep.txt): 0.77 ms per 4K frame against 0.60 ms for the same bytes as
        bare copies (48 GB/s per direction) and 0.42 ms for the device work alone; the driving thread is blocked on the device
        (`pipeline_host_wait_s`) half of the time: copies and kernels do not overlap fully there (a bare
        H2D -> idle kernel -> D2H chain on 8 streams shows the same loss).  Returns (h2d_bytes, d2h_bytes) summed over all jobs."""
        F, H, W, _ = host_in.shape
        J = F * repeat
        lag = min(lag, slots - 1)
        dev = torch.device("cuda", self.device)
        if not hasattr(self, "_streams") or len(self._streams) < slots:
            self._streams = [torch.cuda.Stream(device=dev) for _ in range(slots)]
        self.pipeline_host_wait_s = 0.0                            # time the host spent blocked on the device (diagnostic)
        h2d = d2h = 0
        jobs: List[_Job] = []
        for k in range(J):
            slot = k % slots
            if k >= slots:
                self._wait_decoded(jobs[k - slots])                # the slot's previous job must be done with its buffers
            p = self._plan(1, H, W, space, brange, qrange, instance=slot)
            st = self._host_staging(p)
            src = st.rgb_dev.get(host_in.dtype)
            if src is None:
                src = st.rgb_dev[host_in.dtype] = torch.empty((1, H, W, 3), dtype=host_in.dtype, device=dev)
            f = k % F
            # phase A: upload + encode + counts
            with torch.cuda.stream(self._streams[slot]):
                src.copy_(host_in[f:f + 1], non_blocking=True)
                enc = self.encode(src, space, qrange, brange, instance=slot)
                st.counts.copy_(enc.counts, non_blocking=True)
                if packed:
                    pk = self.pack(enc, space, qrange, brange, instance=slot)
                    st.pk_counts.copy_(pk.counts, non_blocking=True)
                encoded = torch.cuda.Event()
                encoded.record()
            jobs.append(_Job(f, slot, p, enc, encoded))
            h2d += host_in[0].numel() * host_in.element_size()
            # phase B of a job is issued `lag` jobs after its phase A (its counts have landed by then), and a slot is
            # reused only `slots` jobs later, so neither host wait normally blocks
            if k >= lag:
                a, b_ = self._phase_b(jobs[k - lag], host_out, space, qrange, brange, packed)
                h2d += a; d2h += b_
        for jb in jobs[max(0, J - lag):]:
            a, b_ = self._phase_b(jb, host_out, space, qrange, brange, packed)
            h2d += a; d2h += b_
        for jb in jobs[max(0, J - slots):]:
            self._wait_decoded(jb)
        return h2d, d2h

    def _phase_b(self, job: _Job, host_out, space, qrange, brange, packed: bool):
        p, st, enc, slot = job.p, job.p.staging, job.enc, job.slot
        t0 = time.perf_counter()
        job.encoded.synchronize()                                  # counts are on the host now
        self.pipeline_host_wait_s += time.perf_counter() - t0
        counts = st.counts.numpy()[0]
        pkc = st.pk_counts.numpy()[0]
        h2d = d2h = st.counts.numel() * 4
        H, W = p.info.height, p.info.width
        out_kind = "u8" if host_out.dtype == torch.uint8 else "f32"
        route_packed = packed and not pkc[:, 2].any()
        if route_packed:
            arena_dev, arena_host = self._arena(p)
        with torch.cuda.stream(self._streams[slot]):
            if route_packed:
                # gather the job's packed streams into one arena, ONE copy each way, scatter back
                pk = p.packed
                off = 0
                there, back = [], []
                for l in range(3):
                    nl, ns = int(counts[l, 0]), int(counts[l, 1])
                    nnz, nw = int(pkc[l, 0]), int(pkc[l, 3])
                    for t, nb, needed_back in ((pk.mask[l][0], nw * 4, True), (pk.vals[l][0], nnz * 2, True), (enc.leaves[l][0], nl * 16, True),
                                               (enc.states[l][0], ns, False)):
                        there.append((t.data_ptr(), arena_dev.data_ptr() + off, nb))
                        if needed_back:
                            back.append((arena_dev.data_ptr() + off, t.data_ptr(), nb))
                        off = (off + nb + 15) & ~15
                self._copy_segments(there)
                arena_host[:off].copy_(arena_dev[:off], non_blocking=True)          # -> the host-side entropy coder
                arena_dev[:off].copy_(arena_host[:off], non_blocking=True)          # <- what the entropy decoder hands back
                self._copy_segments(back)
                enc.counts.copy_(st.counts, non_blocking=True)
                pk.counts.copy_(st.pk_counts, non_blocking=True)
                self.unpack(pk, 1, H, W, space, qrange, brange, instance=slot)
                h2d += off + 2 * st.counts.numel() * 4
                d2h += off
            else:
                # raw int32 streams (packed=False, or a plane whose coefficients do not fit int16): per-range copies
                for l in range(3):
                    nl, ns, nc = (int(counts[l, i]) for i in range(3))
                    st.coef[l][:nc].copy_(enc.coef[l][0, :nc], non_blocking=True)
                    st.leaves[l][:nl].copy_(enc.leaves[l][0, :nl], non_blocking=True)
                    st.states[l][:ns].copy_(enc.states[l][0, :ns], non_blocking=True)
                    d2h += nc * 4 + nl * 16 + ns
                for l in range(3):
                    nl, nc = int(counts[l, 0]), int(counts[l, 2])
                    enc.coef[l][0, :nc].copy_(st.coef[l][:nc], non_blocking=True)
                    enc.leaves[l][0, :nl].copy_(st.leaves[l][:nl], non_blocking=True)
                    h2d += nc * 4 + nl * 16
                enc.counts.copy_(st.counts, non_blocking=True)
            rgb = self.decode(enc.coef, enc.leaves, enc.counts, 1, H, W, space, qrange, brange, instance=slot, out=out_kind)
            host_out[job.frame:job.frame + 1].copy_(rgb, non_blocking=True)
            d2h += rgb.numel() * rgb.element_size()
            job.decoded = torch.cuda.Event()
            job.decoded.record()
        return h2d, d2h

    def _wait_decoded(self, job: _Job):
        t0 = time.perf_counter()
        job.decoded.synchronize()
        self.pipeline_host_wait_s += time.perf_counter() - t0

    def decode_encoded(self, enc: EncodedBatch, space, qrange, brange, out: str = "f32"):
        B, H, W = enc.shape
        return self.decode(enc.coef, enc.leaves, enc.counts, B, H, W, space, qrange, brange, zigzag=enc.zigzag, out=out)

    # ------------------------------------------------------------------------------------------
    # host <-> device helpers for the reference-facing shim
    # ------------------------------------------------------------------------------------------
    def download(self, enc: EncodedBatch):
        """D2H of exactly the used parts. Returns per image a list of 3 dicts(leaves, states, coef, root)."""
        counts = enc.counts.cpu().numpy()                  # synchronises the stream
        self.check_status(enc.status, "encode")
        B = enc.shape[0]
        out = []
        for b in range(B):
            layers = []
            for l in range(3):
                nl, ns, nc, root = (int(v) for v in counts[b, l])
                d = dict(leaves=enc.leaves[l][b, :nl].cpu().numpy(), states=enc.states[l][b, :ns].cpu().numpy(),
                         coef=enc.coef[l][b, :nc].cpu().numpy(), root=root, zigzag=enc.zigzag)
                if enc.zigzag and enc.packed_states is not None:
                    d["packed_states"] = enc.packed_states[l][b, :(ns + 3) // 4].cpu().numpy()
                layers.append(d)
            out.append(layers)
        return out

    def upload_for_decode(self, per_image_layers, B, H, W, space, qrange, brange):
        """per_image_layers[b][l] = dict(leaves (n,4) int32 incl. coef offsets, coef int32). Returns device buffers."""
        p = self._plan(B, H, W, space, brange, qrange)
        o = p.out
        counts = np.zeros((B, 3, 4), dtype=np.int32)
        for b in range(B):
            for l in range(3):
                d = per_image_layers[b][l]
                nl, nc = len(d["leaves"]), len(d["coef"])
                if nl > p.info.cap_leaves[l] or nc > p.info.cap_coef[l]:
                    raise ValueError("stream does not fit the layer geometry (corrupt input?)")
                counts[b, l, 0] = nl
                counts[b, l, 2] = nc
                o.leaves[l][b, :nl].copy_(torch.from_numpy(np.require(d["leaves"], dtype=np.int32, requirements=["C", "W"])), non_blocking=False)
                o.coef[l][b, :nc].copy_(torch.from_numpy(np.require(d["coef"], dtype=np.int32, requirements=["C", "W"])), non_blocking=False)
        o.counts.copy_(torch.from_numpy(counts))
        return o.coef, o.leaves, o.counts


_codecs: Dict[int, DeviceCodec] = {}


def get_codec(device: Optional[int] = None) -> DeviceCodec:
    _require_cuda()
    if device is None:
        device = torch.cuda.current_device()
    if device not in _codecs:
        _codecs[device] = DeviceCodec(device)
    return _codecs[device]


# ----------------------------------------------------------------------------------------------
# single-plane stage calls (numpy in / numpy out) used by the color / jpeg drop-in modules and tests
# ----------------------------------------------------------------------------------------------
class Stages:
    def __init__(self, device: Optional[int] = None):
        _require_cuda()
        self.device = torch.cuda.current_device() if device is None else device
        self.lib = native.load()
        self.handle = native.handle(self.device)
        self.dev = torch.device("cuda", self.device)

    def _ws(self, h, w, mn=0, mx=0):
        n = self.lib.aeaj_stage_workspace_bytes(h, w, mn, mx)
        return torch.empty(int(n), dtype=torch.uint8, device=self.dev)

    def _to(self, a, dtype):
        return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).to(self.dev)

    def color(self, space: str, x: np.ndarray, inverse: bool) -> np.ndarray:
        t = self._to(x, np.float32)
        o = torch.empty_like(t)
        fn = self.lib.aeaj_color_inverse if inverse else self.lib.aeaj_color_forward
        native.check(fn(self.handle, tables.SPACE_ID[space], t.data_ptr(), o.data_ptr(), t.shape[0], _stream()), "aeaj_color")
        return o.cpu().numpy()

    def normalize(self, space: str, channel: int, x: np.ndarray, inverse: bool) -> np.ndarray:
        t = self._to(x, np.float32)
        o = torch.empty_like(t)
        native.check(self.lib.aeaj_normalize(self.handle, tables.SPACE_ID[space], channel, int(inverse), t.data_ptr(), o.data_ptr(),
                                             t.numel(), _stream()), "aeaj_normalize")
        return o.cpu().numpy()

    def downsample(self, layer: np.ndarray, h: int, w: int) -> np.ndarray:
        t = self._to(layer, np.float32)
        o = torch.empty((h, w), dtype=torch.float32, device=self.dev)
        native.check(self.lib.aeaj_downsample_area(self.handle, t.data_ptr(), t.shape[0], t.shape[1], o.data_ptr(), h, w, _stream()),
                     "aeaj_downsample_area")
        return o.cpu().numpy()

    def resize_linear(self, layer: np.ndarray, H: int, W: int) -> np.ndarray:
        t = self._to(layer, np.float32)
        o = torch.empty((H, W), dtype=torch.float32, device=self.dev)
        native.check(self.lib.aeaj_resize_linear(self.handle, t.data_ptr(), t.shape[0], t.shape[1], o.data_ptr(), H, W, _stream()),
                     "aeaj_resize_linear")
        return o.cpu().numpy()

    def cast_u8(self, layer: np.ndarray) -> np.ndarray:
        t = self._to(layer, np.float32)
        o = torch.empty(t.shape, dtype=torch.uint8, device=self.dev)
        native.check(self.lib.aeaj_cast_u8(self.handle, t.data_ptr(), o.data_ptr(), t.numel(), _stream()), "aeaj_cast_u8")
        return o.cpu().numpy()

    def _u8_stage(self, fn, src: np.ndarray) -> np.ndarray:
        t = self._to(src, np.uint8)
        h, w = t.shape
        o = torch.empty_like(t)
        ws = self._ws(h, w)
        native.check(fn(self.handle, t.data_ptr(), h, w, o.data_ptr(), ws.data_ptr(), _stream()), "u8 stage")
        return o.cpu().numpy()

    def clahe(self, src):
        return self._u8_stage(self.lib.aeaj_clahe, src)

    def gauss3(self, src):
        return self._u8_stage(self.lib.aeaj_gauss3, src)

    def bilateral5(self, src):
        return self._u8_stage(self.lib.aeaj_bilateral5, src)

    def percentile_thresholds(self, src: np.ndarray):
        t = self._to(src, np.uint8)
        h, w = t.shape
        thr = torch.empty(2, dtype=torch.float64, device=self.dev)
        ws = self._ws(h, w)
        native.check(self.lib.aeaj_percentile_thresholds(self.handle, t.data_ptr(), h, w, thr.data_ptr(), ws.data_ptr(), _stream()),
                     "aeaj_percentile_thresholds")
        v = thr.cpu().numpy()
        return float(v[0]), float(v[1])

    def canny_u8(self, src: np.ndarray, lo: float, hi: float) -> np.ndarray:
        t = self._to(src, np.uint8)
        h, w = t.shape
        thr = torch.tensor([lo, hi], dtype=torch.float64, device=self.dev)
        o = torch.empty_like(t)
        ws = self._ws(h, w)
        native.check(self.lib.aeaj_canny_u8(self.handle, t.data_ptr(), h, w, thr.data_ptr(), o.data_ptr(), ws.data_ptr(), _stream()),
                     "aeaj_canny_u8")
        return o.cpu().numpy()

    def canny(self, layer: np.ndarray) -> np.ndarray:
        t = self._to(layer, np.float32)
        h, w = t.shape
        o = torch.empty((h, w), dtype=torch.uint8, device=self.dev)
        ws = self._ws(h, w)
        native.check(self.lib.aeaj_canny(self.handle, t.data_ptr(), h, w, o.data_ptr(), ws.data_ptr(), _stream()), "aeaj_canny")
        return o.cpu().numpy()

    def quadtree(self, edge: np.ndarray, max_size: int, min_size: int):
        """-> (leaves (n,4) int32 x,y,size,coef_off ; states uint8 ; root)"""
        e = np.ascontiguousarray(edge == 1).astype(np.uint8)
        t = self._to(e, np.uint8)
        h, w = t.shape
        cl, cs, cc, root = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int()
        native.check(self.lib.aeaj_quadtree_caps(h, w, min_size, max_size, C.byref(cl), C.byref(cs), C.byref(cc), C.byref(root)),
                     "aeaj_quadtree_caps")
        leaves = torch.empty((cl.value, 4), dtype=torch.int32, device=self.dev)
        states = torch.empty(cs.value, dtype=torch.uint8, device=self.dev)
        counts = torch.zeros(4, dtype=torch.int32, device=self.dev)
        ws = self._ws(h, w, min_size, max_size)
        native.check(self.lib.aeaj_quadtree(self.handle, t.data_ptr(), h, w, min_size, max_size, leaves.data_ptr(), states.data_ptr(),
                                            counts.data_ptr(), ws.data_ptr(), _stream()), "aeaj_quadtree")
        c = counts.cpu().numpy()
        return leaves[: int(c[0])].cpu().numpy(), states[: int(c[1])].cpu().numpy(), int(c[3])

    def _qtab_ptrs(self, tabs: dict):
        arr = (C.c_void_p * 9)()
        keep = []
        for s, m in tabs.items():
            t = self._to(m, np.int32)
            keep.append(t)
            arr[int(np.log2(s))] = t.data_ptr()
        return arr, keep

    def dct_quant(self, layer: np.ndarray, leaves: np.ndarray, tabs: dict, mid: float, scale: float, brange) -> np.ndarray:
        t = self._to(layer, np.float32)
        h, w = t.shape
        lv = self._to(leaves, np.int32)
        n_coef = int((leaves[:, 2].astype(np.int64) ** 2).sum())
        counts = torch.tensor([len(leaves), 0, n_coef, 0], dtype=torch.int32, device=self.dev)
        coef = torch.empty(max(n_coef, 1), dtype=torch.int32, device=self.dev)
        arr, keep = self._qtab_ptrs(tabs)
        ws = self._ws(h, w, brange[0], brange[1])
        native.check(self.lib.aeaj_dct_quant(self.handle, t.data_ptr(), h, w, mid, scale, lv.data_ptr(), counts.data_ptr(), brange[0], brange[1],
                                             arr, coef.data_ptr(), ws.data_ptr(), _stream()), "aeaj_dct_quant")
        return coef[:n_coef].cpu().numpy()

    def dequant_idct(self, coef: np.ndarray, leaves: np.ndarray, tabs: dict, h: int, w: int, mid: float, scale: float, brange) -> np.ndarray:
        cf = self._to(coef, np.int32)
        lv = self._to(leaves, np.int32)
        counts = torch.tensor([len(leaves), 0, len(coef), 0], dtype=torch.int32, device=self.dev)
        out = torch.zeros((h, w), dtype=torch.float32, device=self.dev)
        arr, keep = self._qtab_ptrs(tabs)
        ws = self._ws(h, w, brange[0], brange[1])
        native.check(self.lib.aeaj_dequant_idct(self.handle, cf.data_ptr(), lv.data_ptr(), counts.data_ptr(), brange[0], brange[1], arr, h, w,
                                                mid, scale, out.data_ptr(), ws.data_ptr(), _stream()), "aeaj_dequant_idct")
        return out.cpu().numpy()


_stages: Dict[int, Stages] = {}


def get_stages(device: Optional[int] = None) -> Stages:
    _require_cuda()
    if device is None:
        device = torch.cuda.current_device()
    if device not in _stages:
        _stages[device] = Stages(device)
    return _stages[device]
