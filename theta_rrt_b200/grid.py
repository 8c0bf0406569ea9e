"""Occupancy grids: `builtins.imarray` (main.py:38-42) as a bit-packed device tensor.

Layout (include/thetarrt.h): per map H rows of wpr=(W+31)//32 32-bit words,
pixel (x, y) = bit (x & 31) of word [y*wpr + (x >> 5)], 1 = free, padding = blocked.
Packing runs on the device (trrt_pack_grid).  `tiles` is a derived copy in overlapping 8x16-pixel strips, one set
per driving axis, for the batched line-of-sight kernel (trrt_tile_grid; layout in include/thetarrt.h, K4b).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib


def load_png(path) -> np.ndarray:
    """np.array(Image.open(path).convert('1')) -- exactly main.py:38-42 (incl. PIL's dither for grey images)."""
    from PIL import Image
    return np.array(Image.open(path).convert("1"))


def _int_array(x, what):
    a = np.asarray(x)
    if a.size == 0:
        a = a.astype(np.int64)
    if a.dtype.kind not in "iu":
        raise ValueError(f"{what} must be integers, got {a.dtype}")
    return np.ascontiguousarray(a.astype(np.int64))


class OccupancyGrid:
    """One or several square maps of identical size, resident on one GPU."""

    def __init__(self, free, device="cuda:0"):
        free = np.asarray(free)
        if free.ndim == 2:
            free = free[None]
        if free.ndim != 3:
            raise ValueError("free must be (H, W) or (n_maps, H, W)")
        self.n_maps, self.H, self.W = (int(s) for s in free.shape)
        if self.H != self.W:
            raise ValueError("maps must be square: the reference's bounds test (search.py:21) compares x with "
                             "shape[0] and y with shape[1]")
        self.device = torch.device(device)
        lib = _lib.load()
        self.wpr = (self.W + 31) // 32
        words = self.n_maps * lib.trrt_grid_words(self.H, self.W)
        with torch.cuda.device(self.device):
            d_free = torch.from_numpy(np.ascontiguousarray(free.astype(bool).astype(np.uint8))).to(self.device)
            self.bits = torch.empty(words, dtype=torch.int32, device=self.device)
            st = torch.cuda.current_stream(self.device).cuda_stream
            _lib.check(lib.trrt_pack_grid(d_free.data_ptr(), self.n_maps, self.H, self.W, self.bits.data_ptr(), st),
                       "trrt_pack_grid")
            torch.cuda.current_stream(self.device).synchronize()  # d_free may be freed after return
        self.nbytes = words * 4
        self._tiles = None

    @property
    def tiles(self):
        """Strip copy of the grid (include/thetarrt.h K4b, 4x the packed rows), built on first use by trrt_tile_grid
        from the packed rows."""
        if self._tiles is None:
            lib = _lib.load()
            with torch.cuda.device(self.device):
                t = torch.empty(self.n_maps * lib.trrt_tile_words(self.H, self.W), dtype=torch.int64, device=self.device)
                st = torch.cuda.current_stream(self.device).cuda_stream
                _lib.check(lib.trrt_tile_grid(self.bits.data_ptr(), self.n_maps, self.H, self.W, t.data_ptr(), st),
                           "trrt_tile_grid")
                self._tiles_ready = torch.cuda.Event()
                self._tiles_ready.record(torch.cuda.current_stream(self.device))
            self._tiles = t
        else:  # built on some stream earlier: the caller's stream must not run ahead of that build
            torch.cuda.current_stream(self.device).wait_event(self._tiles_ready)
        return self._tiles

    def edit(self, rects, free, map_id=None):
        """imarray[y0:y1, x0:x1] = free for every rectangle, in place on the device (trrt_grid_edit), enqueued on the
        current stream.  rects: int [n, 4] = (x0, y0, x1, y1), pixels x0 <= x < x1, y0 <= y < y1 (a pixel is a 1x1
        rectangle); they are clipped to the image (no negative indexing) and empty ones do nothing.  free: bool, one for
        all or [n].  map_id: None (map 0), one int, or [n].  A pixel that a free and a blocked rectangle of one call both
        cover ends blocked.  Host rects must fit int32, and map ids outside [0, n_maps) raise ValueError; rects and map
        ids in CUDA tensors are not read on the host, must be int32, and map ids outside [0, n_maps) are ignored.
        When the strip copy (`tiles`) exists, only its entries that the rectangles touch are rebuilt, and streams that use
        `tiles` later wait for the patch.  Kernels that read the grid on other streams are the caller's to order, as for
        any in-place write to a tensor."""
        r = rects if isinstance(rects, torch.Tensor) else torch.from_numpy(_int_array(rects, "rects"))
        if r.numel() == 0:
            r = r.reshape(0, 4)
        if r.dim() != 2 or r.shape[1] != 4:
            raise ValueError("rects must be [n, 4] = (x0, y0, x1, y1)")
        if r.is_floating_point() or r.dtype == torch.bool:
            raise ValueError(f"rects must be integers, got {r.dtype}")
        if r.is_cuda and r.dtype != torch.int32:  # not read on the host, so not narrowed either
            raise ValueError(f"rects in a CUDA tensor must be int32, got {r.dtype}")
        n = r.shape[0]
        if not r.is_cuda and n and (int(r.min()) < -2 ** 31 or int(r.max()) >= 2 ** 31):
            raise ValueError("rect coordinates must fit int32")
        if map_id is None:
            mid = torch.zeros(n, dtype=torch.int32)
        elif isinstance(map_id, torch.Tensor) and map_id.is_cuda:
            if map_id.dtype != torch.int32:
                raise ValueError(f"map ids in a CUDA tensor must be int32, got {map_id.dtype}")
            mid = map_id.reshape(-1).expand(n) if map_id.numel() == 1 else map_id.reshape(-1)
        else:
            m = _int_array(map_id, "map_id").reshape(-1)
            if m.size and (int(m.min()) < 0 or int(m.max()) >= self.n_maps):
                raise ValueError(f"map ids must lie in [0, {self.n_maps})")
            mid = torch.from_numpy(np.full(n, m[0], np.int64) if m.size == 1 else m)
        fr = free if isinstance(free, torch.Tensor) else torch.from_numpy(np.asarray(free, dtype=bool))
        fr = fr.reshape(-1).expand(n) if fr.numel() == 1 else fr.reshape(-1)
        if mid.numel() != n or fr.numel() != n:
            raise ValueError(f"{n} rects need one free flag / map id each, or one for all")
        lib = _lib.load()
        with torch.cuda.device(self.device):
            d_rects = torch.cat([r.to(self.device, torch.int32), mid.to(self.device, torch.int32)[:, None]], dim=1).contiguous()
            d_free = fr.to(self.device, torch.uint8).contiguous()
            stream = torch.cuda.current_stream(self.device)
            tiles = self._tiles
            if tiles is not None:
                stream.wait_event(self._tiles_ready)
            _lib.check(lib.trrt_grid_edit(self.bits.data_ptr(), tiles.data_ptr() if tiles is not None else None, self.n_maps,
                                          self.H, self.W, d_rects.data_ptr(), d_free.data_ptr(), n, stream.cuda_stream),
                       "trrt_grid_edit")
            if tiles is not None:
                self._tiles_ready = torch.cuda.Event()
                self._tiles_ready.record(stream)

    @property
    def shape(self):
        return (self.H, self.W)
