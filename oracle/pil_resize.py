"""NumPy restatement of the reference's crop transform up to T.ToTensor():

    img.rotate(rotation, expand=True)  ->  T.Resize(img_size, BICUBIC)        (strhub/data/module.py:69-82)

On a PIL image torchvision's Resize is `PIL.Image.resize((W, H), BICUBIC)`, and PIL's resampler is a deterministic
separable filter (libImaging/Resample.c): coefficients in double precision (precompute_coeffs / bicubic_filter, a = -0.5),
quantised to int32 with 22 fraction bits (normalize_coeffs_8bpc), integer sums clipped to uint8 after each pass,
horizontal pass first - except for images more than 100 times taller than wide, which Image.resize shrinks vertically
first (`vertical_first`).  An axis whose size does not change is not resampled.  Python / NumPy float64 arithmetic is IEEE
double without contraction, so this restatement is bit-exact, and so is the CUDA kernel that follows the same expression
order (parseq_b200/csrc/resize.cuh).  For multiples of 90 degrees, `rotate(expand=True)` is an exact transpose.

    python -m oracle.pil_resize      # writes tests/golden/crops/resize.pt (needs no PIL)
"""
from __future__ import annotations

import os
from typing import List, Tuple

import numpy as np

PRECISION_BITS = 22
MAX_SIDE = 4096
ROTATIONS = (0, 90, 180, 270)


def bicubic_filter(x: np.ndarray) -> np.ndarray:
    """Resample.c bicubic_filter with a = -0.5, same operation order."""
    a = -0.5
    x = np.abs(x)
    inner = ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    outer = (((x - 5) * x + 8) * x - 4) * a
    return np.where(x < 1.0, inner, np.where(x < 2.0, outer, 0.0))


def precompute_coeffs(in_size: int, out_size: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """(xmin [out], count [out], int32 weights [out, ksize]) as Resample.c precompute_coeffs + normalize_coeffs_8bpc."""
    scale = float(in_size) / out_size
    filterscale = max(scale, 1.0)
    support = 2.0 * filterscale
    ksize = int(np.ceil(support)) * 2 + 1
    ss = 1.0 / filterscale
    xmins = np.zeros(out_size, np.int64)
    counts = np.zeros(out_size, np.int64)
    kk = np.zeros((out_size, ksize), np.int64)
    for xx in range(out_size):
        center = 0.0 + (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)          # C casts truncate toward zero, like int()
        xmax = min(int(center + support + 0.5), in_size) - xmin
        w = bicubic_filter((np.arange(xmax, dtype=np.float64) + xmin - center + 0.5) * ss)
        ww = 0.0
        for v in w:                                          # sequential sum, as in C
            ww += float(v)
        if ww != 0.0:
            w = w / ww
        q = w * (1 << PRECISION_BITS)
        kk[xx, :xmax] = np.where(w < 0, (-0.5 + q), (0.5 + q)).astype(np.int64)   # astype truncates toward zero
        xmins[xx], counts[xx] = xmin, xmax
    return xmins, counts, kk


def _clip8(acc: np.ndarray) -> np.ndarray:
    return np.clip(acc >> PRECISION_BITS, 0, 255).astype(np.uint8)


def _resample_axis1(img: np.ndarray, out_size: int) -> np.ndarray:
    """Resample axis 1 of an int [rows, in, ch] array."""
    xmins, counts, kk = precompute_coeffs(img.shape[1], out_size)
    src = img.astype(np.int64)
    out = np.empty((img.shape[0], out_size, img.shape[2]), np.uint8)
    for xx in range(out_size):
        n, x0 = counts[xx], xmins[xx]
        acc = np.full((img.shape[0], img.shape[2]), 1 << (PRECISION_BITS - 1), np.int64)
        acc += np.einsum("rkc,k->rc", src[:, x0:x0 + n], kk[xx, :n])
        out[:, xx] = _clip8(acc)
    return out


def rotate(img: np.ndarray, rotation: int) -> np.ndarray:
    """PIL `Image.rotate(rotation, expand=True)` for rotation in {0, 90, 180, 270} (counter-clockwise)."""
    if rotation not in ROTATIONS:
        raise ValueError(f"rotation must be one of {ROTATIONS}, got {rotation}")
    return np.ascontiguousarray(np.rot90(img, k=rotation // 90))


def vertical_first(h: int, w: int, H: int) -> bool:
    """Image.resize resizes an image more than 100 times taller than wide in two calls, height first, when the height
    shrinks; otherwise one call, horizontal pass first."""
    return h > w * 100 and H < h


def resize(img: np.ndarray, size: Tuple[int, int]) -> np.ndarray:
    """PIL `Image.resize((W, H), BICUBIC)` of a uint8 [h, w, 3] array; size = (H, W)."""
    H, W = size
    out = np.asarray(img, dtype=np.uint8)
    vfirst = vertical_first(out.shape[0], out.shape[1], H)
    if vfirst:
        out = _resample_axis1(out.transpose(1, 0, 2), H).transpose(1, 0, 2)
    if out.shape[1] != W:
        out = _resample_axis1(out, W)
    if out.shape[0] != H:
        out = _resample_axis1(out.transpose(1, 0, 2), H).transpose(1, 0, 2)
    return np.ascontiguousarray(out)


def transform(img: np.ndarray, size: Tuple[int, int], rotation: int = 0) -> np.ndarray:
    """rotate(expand=True) then Resize(size, BICUBIC): uint8 [H, W, 3], what T.ToTensor() receives."""
    return resize(rotate(img, rotation), size)


# ------------------------------------------------------------------------------------------------- golden crops
TARGETS = [(32, 128), (224, 224), (48, 160)]   # PARSeq, ViTSTR / patch16, the ViT-B-width stress configuration


def _content(rng: np.random.Generator, h: int, w: int, smooth: bool) -> np.ndarray:
    if not smooth:
        return rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
    # steps between 0 and 255 with flat runs: bicubic overshoot drives the sums past both clip limits
    yy, xx = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    phase = rng.uniform(0, 6.28, size=3)
    per = rng.uniform(3, 17, size=3)
    ch = [np.where(np.sin((xx + yy * 0.7) / per[c] + phase[c]) > 0, 255, 0) for c in range(3)]
    return np.stack(ch, -1).astype(np.uint8)


def golden_crops(seed: int = 0) -> List[dict]:
    """Seeded crops over the size classes the kernel must cover: (name, image, rotation)."""
    rng = np.random.default_rng(seed)
    sizes = [("1x1", 1, 1), ("identity", 32, 128), ("width_only", 32, 300), ("height_only", 90, 128),
             ("up_both", 8, 20), ("down_both", 200, 900), ("mixed_a", 48, 60), ("mixed_b", 20, 600),
             ("tall", 4096, 16), ("wide", 16, 4096), ("huge", 4096, 4096), ("odd", 33, 129),
             ("tall_narrow", 1500, 12)]
    out = []
    for name, h, w in sizes:
        for smooth in (False, True):
            if name == "huge" and smooth:
                continue
            out.append(dict(name=f"{name}_{'smooth' if smooth else 'random'}", image=_content(rng, h, w, smooth),
                            rotation=0))
    for rot in (90, 180, 270):
        for name, h, w in (("rot_a", 24, 70), ("rot_b", 130, 40), ("rot_wide", 12, 1500)):
            out.append(dict(name=f"{name}_{rot}", image=_content(rng, h, w, rot == 180), rotation=rot))
    return out


def digest(a: np.ndarray) -> str:
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.uint8).tobytes()).hexdigest()


def make_golden(path: str) -> None:
    """The crops are regenerated from their seed (a 4096 x 4096 crop is 48 MB); the file pins their bytes and PIL's
    output for every target size by SHA-256, and keeps the 32 x 128 outputs themselves."""
    import torch
    cases = golden_crops()
    data = dict(names=[c["name"] for c in cases], rotations=[c["rotation"] for c in cases],
                shapes=[tuple(c["image"].shape) for c in cases], inputs=[digest(c["image"]) for c in cases],
                targets=TARGETS, outputs={}, resized_32x128=[])
    for size in TARGETS:
        res = [transform(c["image"], size, c["rotation"]) for c in cases]
        data["outputs"][size] = [digest(r) for r in res]
        if size == (32, 128):
            data["resized_32x128"] = [torch.from_numpy(r) for r in res]
    torch.save(data, path)


if __name__ == "__main__":
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = os.path.join(root, "tests", "golden", "crops", "resize.pt")
    make_golden(p)
    print(p, os.path.getsize(p), "bytes")
