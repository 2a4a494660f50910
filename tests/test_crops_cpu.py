"""Variable-size crop input, CPU side: the NumPy restatement of PIL's rotate + bicubic resize (oracle/pil_resize.py)
against the committed goldens and, where PIL imports, against PIL itself; the packing helper's descriptors; input
validation in Python."""
import os

import numpy as np
import pytest
import torch

from oracle import pil_resize as R

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "crops", "resize.pt")


@pytest.fixture(scope="module")
def golden():
    return torch.load(GOLDEN, weights_only=False)


def test_oracle_equals_goldens(golden):
    cases = R.golden_crops()
    assert [c["name"] for c in cases] == golden["names"]
    for i, c in enumerate(cases):
        assert tuple(c["image"].shape) == tuple(golden["shapes"][i])
        assert R.digest(c["image"]) == golden["inputs"][i], c["name"]       # the seeded generator is unchanged
        assert c["rotation"] == golden["rotations"][i]
    for size in golden["targets"]:
        for i, c in enumerate(cases):
            out = R.transform(c["image"], size, c["rotation"])
            assert out.shape == (size[0], size[1], 3)
            assert R.digest(out) == golden["outputs"][size][i], (c["name"], size)
            if size == (32, 128):
                assert np.array_equal(out, golden["resized_32x128"][i].numpy())


def test_goldens_cover_the_size_classes(golden):
    names = " ".join(golden["names"])
    for cls in ("1x1", "identity", "width_only", "height_only", "up_both", "down_both", "mixed_a", "mixed_b", "tall",
                "wide", "huge", "odd", "tall_narrow", "_smooth", "_random", "_90", "_180", "_270"):
        assert cls in names, cls
    # at least one crop takes PIL's height-first route after rotation, and one without
    shapes = [R.rotate(np.zeros(s, np.uint8), r).shape for s, r in zip(golden["shapes"], golden["rotations"])]
    assert sum(R.vertical_first(h, w, 32) for h, w, _ in shapes) >= 2


def _pil_transform(img, size, rotation):
    from PIL import Image
    im = Image.fromarray(img)
    if rotation:
        im = im.rotate(rotation, expand=True)
    return np.asarray(im.resize((size[1], size[0]), Image.BICUBIC))


@pytest.mark.parametrize("seed", [0, 1])
def test_oracle_equals_live_pil(seed):
    pytest.importorskip("PIL")
    rng = np.random.default_rng(1000 + seed)
    sizes = [(int(rng.integers(1, 200)), int(rng.integers(1, 700))) for _ in range(12)]
    sizes += [(1, 1), (32, 128), (31, 500), (100, 40), (33, 129), (2100, 12), (9, 1500)]
    for k, (h, w) in enumerate(sizes):
        img = R._content(rng, h, w, smooth=bool(k % 2))
        rot = R.ROTATIONS[k % 4]
        for size in R.TARGETS:
            assert np.array_equal(R.transform(img, size, rot), _pil_transform(img, size, rot)), ((h, w), rot, size)


def test_oracle_equals_torchvision_resize():
    pytest.importorskip("PIL")
    T = pytest.importorskip("torchvision.transforms")
    from PIL import Image
    rng = np.random.default_rng(7)
    for h, w in [(20, 90), (64, 300), (5, 7), (1800, 15)]:
        img = R._content(rng, h, w, smooth=False)
        got = np.asarray(T.Resize((32, 128), T.InterpolationMode.BICUBIC)(Image.fromarray(img)))
        assert np.array_equal(R.transform(img, (32, 128)), got)


def _bytes_of(packed, i):
    buf = packed.keepalive[0].reshape(-1)
    d = packed.desc[i]
    rows = [buf[d.offset + r * d.row_stride: d.offset + r * d.row_stride + 3 * d.width] for r in range(d.height)]
    return torch.stack(rows).reshape(d.height, d.width, 3).numpy()


def test_pack_numpy_pil_and_tensors():
    from parseq_b200.crops import pack_crops
    rng = np.random.default_rng(3)
    a = rng.integers(0, 256, (5, 7, 3), dtype=np.uint8)
    frame = torch.from_numpy(rng.integers(0, 256, (40, 60, 3), dtype=np.uint8))
    view = frame[3:13, 20:45]                                   # row stride 180 bytes, not contiguous
    items = [a, view, frame[0:1, 0:1]]
    try:
        from PIL import Image
        items.append(Image.fromarray(a[:, :4].copy()).convert("L"))   # converted to RGB like read.py
    except ImportError:
        pass
    p = pack_crops(items, rotation=270, pin_memory=False)
    assert p.host and p.count == len(items) and p.rotation == 270
    off = 0
    for i, it in enumerate(items):
        d = p.desc[i]
        ref = np.asarray(it.convert("RGB")) if not isinstance(it, (np.ndarray, torch.Tensor)) else np.asarray(it)
        assert (d.offset, d.height, d.width, d.row_stride) == (off, ref.shape[0], ref.shape[1], 3 * ref.shape[1])
        assert np.array_equal(_bytes_of(p, i), ref)
        off += ref.size
    assert p.pixels_bytes == off
    assert pack_crops([], pin_memory=False).count == 0


@pytest.mark.parametrize("bad, msg", [
    (np.zeros((4, 4, 3), np.float32), "uint8"),
    (np.zeros((4, 4, 4), np.uint8), "RGB"),
    (np.zeros((4, 4), np.uint8), "RGB"),
    (np.zeros((0, 5, 3), np.uint8), "empty"),
    (np.zeros((4097, 2, 3), np.uint8), "4096"),
    (torch.zeros((3, 3, 3), dtype=torch.int16), "uint8"),
    ("not an image", "expected"),
])
def test_pack_rejects_bad_crops(bad, msg):
    from parseq_b200.crops import pack_crops
    with pytest.raises((TypeError, ValueError), match=msg):
        pack_crops([np.zeros((2, 2, 3), np.uint8), bad], pin_memory=False)


def test_pack_rejects_bad_rotation():
    from parseq_b200.crops import pack_crops
    with pytest.raises(ValueError, match="rotation"):
        pack_crops([np.zeros((2, 2, 3), np.uint8)], rotation=45, pin_memory=False)
