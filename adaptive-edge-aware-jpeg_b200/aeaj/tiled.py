"""Halo-split of ONE large image over G GPUs of one node (SURVEY.md 8e, BASELINE config C4).

Rank r owns the band of full-resolution rows [r*H/G, (r+1)*H/G) (a multiple of 256 rows, so no chroma cell, filter
tile or quadtree leaf straddles two ranks).  Everything heavy is sharded -- colour, CLAHE histograms, the fused
prefilter, Sobel / NMS, the quadtree and the DCT -- and nothing on the data path goes through a collective library:

  * the ranks share their plan workspaces through CUDA IPC (``aeaj_peer_*``): a buffer at offset o of this rank's
    workspace is at offset o of every peer's, so the stencil kernels read the 3 / 2 / 1 halo rows outside their band
    straight from the neighbour GPU over NVLink, and the CLAHE / percentile kernels sum the per-rank partial
    histograms on the fly;
  * between phases the ranks meet at a device-side barrier (one tiny kernel per rank that stores an epoch into every
    peer's flag array and spins on its own, ordered with the data by the stream);
  * two small gathers copy the other bands' rows of the strong / weak bitmaps (the hysteresis fixed point is global;
    at 0.15 ms per 64 MP it runs replicated) and of the quadtree block totals (the scan over all top blocks needs
    them; counting and emitting are sharded).

    barrier                                   (the previous call's readers are done with this rank's planes)
    colour + subsample + u8 cast (band), CLAHE histograms (band)
    barrier
    CLAHE LUT (sum of partial histograms) + Gaussian + bilateral (band; 3 halo rows from the neighbours)
    barrier
    thresholds (sum of partial histograms) + Sobel / NMS (band; 2 halo rows)
    barrier,  gather strong / weak rows,  hysteresis (whole image, replicated)
    quadtree counts (band),  barrier,  gather block totals,  scan + emit (band)
    DCT + quantise (band's leaves, coefficients at their global offsets)

Decode: IDCT per band, barrier, upsample (1 chroma halo row from the neighbour) + inverse colour per band.
The library holds this schedule (``aeaj_encode_halo`` / ``aeaj_decode_halo``, one call per direction).  Every rank
ends with its band's leaves / states / coefficients at their global positions of the reference-ordered streams,
bit-identical to the single-GPU result (tests/multi_gpu_halo.py, bench.py's C4 leg).

``emulate=G`` runs the same library schedule for all G bands on ONE GPU, band after band within each phase (the
buffers are shared, so the barriers and gathers are no-ops); the GPU tests use it to check the band-restricted kernels.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import native
from .codec import DeviceCodec, EncodedBatch, _stream

BAND_ALIGN = 256


def band_of(rank: int, world: int, H: int, block_max: int = 128):
    """rows [lo, hi) of the full-resolution image owned by `rank` (bands are multiples of 2 x max(128, block_max) rows)"""
    align = max(BAND_ALIGN, 2 * block_max)
    if H % (world * align) != 0:
        raise ValueError(f"halo-split needs the image height ({H}) to be a multiple of {align} x world size ({world})")
    hb = H // world
    return rank * hb, (rank + 1) * hb


class _Peers:
    """the shared workspace of one plan and its mappings into this process"""

    def __init__(self, lib, plan, rank, world, group):
        import torch.distributed as dist
        self.lib, self.world = lib, world
        self.plan_ptr = plan.ptr.value
        nbytes = int(plan.info.workspace_bytes)
        self.ws, self.flags = C.c_void_p(), C.c_void_p()
        native.check(lib.aeaj_peer_alloc(nbytes, C.byref(self.ws)), "aeaj_peer_alloc")
        native.check(lib.aeaj_peer_alloc(256, C.byref(self.flags)), "aeaj_peer_alloc")
        h = (C.c_ubyte * 64)()
        mine = []
        for ptr in (self.ws, self.flags):
            native.check(lib.aeaj_peer_export(ptr, h), "aeaj_peer_export")
            mine.append(bytes(h))
        every = [None] * world
        dist.all_gather_object(every, mine, group=group)
        self.opened = []
        ws_ptrs, fl_ptrs = (C.c_void_p * world)(), (C.c_void_p * world)()
        for r in range(world):
            if r == rank:
                ws_ptrs[r], fl_ptrs[r] = self.ws.value, self.flags.value
                continue
            for k, arr in ((0, ws_ptrs), (1, fl_ptrs)):
                ptr = C.c_void_p()
                native.check(lib.aeaj_peer_open(C.create_string_buffer(every[r][k], 64), C.byref(ptr)), "aeaj_peer_open")
                arr[r] = ptr.value
                self.opened.append(ptr)
        native.check(lib.aeaj_plan_set_peers(plan.ptr, rank, world, ws_ptrs, fl_ptrs), "aeaj_plan_set_peers")
        dist.barrier(group=group)                        # every rank has mapped every workspace before anyone starts

    def close(self):
        for ptr in self.opened:
            self.lib.aeaj_peer_close(ptr)
        self.opened = []
        self.lib.aeaj_peer_free(self.ws)
        self.lib.aeaj_peer_free(self.flags)


class TiledCodec:
    def __init__(self, codec: DeviceCodec, rank: int = 0, world: int = 1, group=None, emulate: int = 0):
        self.codec, self.rank, self.world, self.group, self.emulate = codec, rank, world, group, emulate
        self.lib = codec.lib
        self._peers = {}

    # -- shared workspace --------------------------------------------------------------------------
    def _ws(self, p):
        """device address of the plan workspace the halo calls use (the shared allocation when the ranks are real GPUs)"""
        if self.world <= 1 or self.emulate:
            return p.workspace.data_ptr()
        key = id(p)
        pe = self._peers.get(key)
        if pe is not None and pe.plan_ptr != p.ptr.value:          # the codec evicted / rebuilt that plan: the mapping is stale
            pe.close()
            pe = None
        if pe is None:
            pe = self._peers[key] = _Peers(self.lib, p, self.rank, self.world, self.group)
        return pe.ws.value

    def close(self):
        torch.cuda.synchronize()
        for pe in self._peers.values():
            pe.close()
        self._peers = {}

    def check(self, H, W, space, qrange, brange):
        """raise if a kernel of the last encode / decode of this geometry reported a problem (synchronises)"""
        p = self.codec._plan(1, H, W, space, brange, qrange)
        self.codec.check_status(p.out.status, "encode")

    def _reduce(self, t: torch.Tensor):
        import torch.distributed as dist
        dist.all_reduce(t, group=self.group)

    def _band(self, H: int, brange):
        """(number of bands, first row of this process's band): every band in emulation, this rank's otherwise"""
        G = self.emulate or self.world
        return G, band_of(0 if self.emulate else self.rank, G, H, brange[1])[0]

    # -- encode ---------------------------------------------------------------------------------
    def encode(self, rgb: torch.Tensor, H: int, W: int, space: str, qrange, brange, exchange_coef: bool = False) -> EncodedBatch:
        """rgb: float32 CUDA tensor.  Real multi-rank mode: this rank's band [Hb, W, 3].  Emulation: the whole [H, W, 3].
        Every rank ends with counts for the whole image and with the leaves / states / coefficients of its own band at
        their global positions in the (zero-initialised by the caller, if it wants to sum them) streams.  `exchange_coef`
        sums the streams over the ranks so that every rank holds all of them (parity checks only; NCCL, not timed)."""
        c = self.codec
        p = c._plan(1, H, W, space, brange, qrange)
        o = p.out
        io = native.EncodeIO()
        for l in range(3):
            io.coef[l], io.leaves[l], io.states[l] = o.coef[l].data_ptr(), o.leaves[l].data_ptr(), o.states[l].data_ptr()
        io.counts, io.status = o.counts.data_ptr(), o.status.data_ptr()
        ws = self._ws(p)
        G, lo = self._band(H, brange)
        rgb = rgb.contiguous()
        # the kernel indexes rows from the top of the full image: hand it the (virtual) address of row 0
        io.rgb = rgb.data_ptr() - lo * W * 12
        multi = not self.emulate and self.world > 1
        if multi and exchange_coef:
            for l in range(3):
                o.coef[l].zero_(); o.leaves[l].zero_(); o.states[l].zero_()
        # the plan is shared with DeviceCodec.encode for B = 1: set what it may have left behind (stream layout, tensor mask)
        native.check(self.lib.aeaj_plan_set_stream_layout(p.ptr, 0), "aeaj_plan_set_stream_layout")
        native.check(self.lib.aeaj_plan_set_tensor_dct(p.ptr, c._tensor_mask()), "aeaj_plan_set_tensor_dct")
        o.zigzag = False
        native.check(self.lib.aeaj_encode_halo(p.ptr, C.byref(io), ws, _stream(), G), "aeaj_encode_halo")
        if multi and exchange_coef:
            import torch.distributed as dist
            for l in range(3):
                # sharded quadtree: every rank wrote only its band's leaves / states (zero elsewhere: sum); the all-split levels
                # above the top blocks and the absent nodes are written by every rank with the same value: maximum
                self._reduce(o.leaves[l])
                dist.all_reduce(o.states[l], op=dist.ReduceOp.MAX, group=self.group)
                self._reduce(o.coef[l])
        return o

    # -- decode ---------------------------------------------------------------------------------
    def decode(self, enc: EncodedBatch, H: int, W: int, space: str, qrange, brange) -> torch.Tensor:
        """Returns the full [H, W, 3] buffer; in real multi-rank mode only this rank's band rows are valid."""
        c = self.codec
        p = c._plan(1, H, W, space, brange, qrange)
        io = native.DecodeIO()
        for l in range(3):
            io.coef[l], io.leaves[l] = enc.coef[l].data_ptr(), enc.leaves[l].data_ptr()
        io.counts, io.rgb = enc.counts.data_ptr(), p.rgb_out.data_ptr()
        ws = self._ws(p)
        G, _ = self._band(H, brange)
        native.check(self.lib.aeaj_plan_set_stream_layout(p.ptr, int(enc.zigzag)), "aeaj_plan_set_stream_layout")
        native.check(self.lib.aeaj_plan_set_tensor_dct(p.ptr, c._tensor_mask()), "aeaj_plan_set_tensor_dct")
        native.check(self.lib.aeaj_decode_halo(p.ptr, C.byref(io), ws, _stream(), G), "aeaj_decode_halo")
        return p.rgb_out[0]
