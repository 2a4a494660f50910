"""Packing of variable-size RGB crops for the engine's crop entry points (parseq_forward_crops & co.).

A caller holds crops as PIL images (converted with `.convert("RGB")`, as the reference's read.py does), uint8 numpy
arrays [h, w, 3], or uint8 torch tensors [h, w, 3] on the CPU or a CUDA device.  `pack_crops` turns them into one
pixel buffer plus one descriptor (offset, height, width, row stride in bytes) per crop:
  - CPU inputs are copied into one pinned host buffer (the engine uploads it: parseq_forward_host_crops);
  - CUDA tensors that are views of one storage with pixel stride 3 and channel stride 1 (crops of one frame, any row
    stride) are passed as that storage's address plus offsets, without a copy;
  - other CUDA tensors are packed with one device `cat`.
Bad input raises ValueError / TypeError here, before anything reaches the engine.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Any, List, Optional, Sequence

import numpy as np
import torch

from .engine import CropC, CropsC

MAX_SIDE = 4096
ROTATIONS = (0, 90, 180, 270)


@dataclass
class PackedCrops:
    count: int
    rotation: int
    host: bool                        # pixels in host memory (the _host entry point) or on `device`
    pixels_ptr: int
    pixels_bytes: int
    desc: Any                         # ctypes array of CropC [count]
    device: Optional[torch.device] = None
    keepalive: List[Any] = field(default_factory=list)

    def c_struct(self) -> CropsC:
        return CropsC(self.count, C.cast(self.desc, C.POINTER(CropC)), self.pixels_ptr or None, self.pixels_bytes,
                      self.rotation)

    def sizes(self):
        return [(d.height, d.width) for d in self.desc]


def _is_pil(x) -> bool:
    try:
        from PIL import Image
    except ImportError:
        return False
    return isinstance(x, Image.Image)


def _check_shape(i: int, shape, dtype_ok: bool, dtype) -> None:
    if not dtype_ok:
        raise TypeError(f"crop {i}: dtype must be uint8, got {dtype}")
    if len(shape) != 3 or shape[2] != 3:
        raise ValueError(f"crop {i}: expected an RGB array [height, width, 3], got shape {tuple(shape)}")
    h, w = int(shape[0]), int(shape[1])
    if h < 1 or w < 1:
        raise ValueError(f"crop {i}: empty crop {h}x{w}")
    if h > MAX_SIDE or w > MAX_SIDE:
        raise ValueError(f"crop {i}: {h}x{w} exceeds the maximum side of {MAX_SIDE} pixels")


def _normalise(i: int, c):
    if _is_pil(c):
        c = np.asarray(c.convert("RGB"))
    if isinstance(c, np.ndarray):
        _check_shape(i, c.shape, c.dtype == np.uint8, c.dtype)
        return c
    if isinstance(c, torch.Tensor):
        _check_shape(i, c.shape, c.dtype == torch.uint8, c.dtype)
        return c
    raise TypeError(f"crop {i}: expected a PIL image, a numpy array or a torch tensor, got {type(c).__name__}")


def pack_crops(crops: Sequence[Any], rotation: int = 0, pin_memory: Optional[bool] = None) -> PackedCrops:
    if rotation not in ROTATIONS:
        raise ValueError(f"rotation must be one of {ROTATIONS} (counter-clockwise degrees), got {rotation}")
    items = [_normalise(i, c) for i, c in enumerate(crops)]
    n = len(items)
    desc = (CropC * max(n, 1))()
    on_cuda = [isinstance(t, torch.Tensor) and t.is_cuda for t in items]
    if n and all(on_cuda):
        dev = items[0].device
        if any(t.device != dev for t in items):
            raise ValueError("CUDA crops must all be on one device")
        base = items[0].untyped_storage().data_ptr()
        shared = all(t.untyped_storage().data_ptr() == base and t.stride(2) == 1 and t.stride(1) == 3 and
                     t.stride(0) >= 3 * t.shape[1] and t.stride(0) < 2 ** 31 for t in items)
        if shared:                                       # views into one frame: no copy
            storage = items[0].untyped_storage()
            for i, t in enumerate(items):
                desc[i] = CropC(t.data_ptr() - base, t.shape[0], t.shape[1], t.stride(0), 0)
            return PackedCrops(n, rotation, False, base, storage.nbytes(), desc, dev, [items[0], desc])
        flat = [t.contiguous().reshape(-1) for t in items]
        buf = torch.cat(flat)
        off = 0
        for i, t in enumerate(items):
            desc[i] = CropC(off, t.shape[0], t.shape[1], 3 * t.shape[1], 0)
            off += flat[i].numel()
        return PackedCrops(n, rotation, False, buf.data_ptr(), buf.numel(), desc, dev, [buf, desc])
    if any(on_cuda):
        raise ValueError("crops must be all on the CPU or all on one CUDA device")
    total = sum(int(a.shape[0]) * int(a.shape[1]) * 3 for a in items)
    if pin_memory is None:
        pin_memory = torch.cuda.is_available()
    buf = torch.empty(max(total, 1), dtype=torch.uint8, pin_memory=pin_memory)
    off = 0
    for i, a in enumerate(items):
        h, w = int(a.shape[0]), int(a.shape[1])
        dst = buf[off:off + h * w * 3].view(h, w, 3)
        if isinstance(a, torch.Tensor):
            dst.copy_(a)
        else:
            np.copyto(dst.numpy(), a)
        desc[i] = CropC(off, h, w, 3 * w, 0)
        off += h * w * 3
    return PackedCrops(n, rotation, True, buf.data_ptr() if n else 0, total, desc, None, [buf, desc])
