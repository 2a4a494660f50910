"""Variable-size crop input on the GPU: parseq_resize_crops is byte-exact with PIL (goldens + oracle) for every size
class, rotation and target size, and the crop entry points return exactly what the uint8 entry points return on the
PIL-resized stack."""
import os

import numpy as np
import pytest
import torch

from oracle import pil_resize as R

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "crops", "resize.pt")
EXPERIMENT_OF_SIZE = {(32, 128): "parseq", (224, 224): "parseq-patch16-224", (48, 160): "parseq-base-48x160"}


def _model(experiment, seed=0, **kw):
    from parseq_b200.config import make_config
    from parseq_b200.factory import create_model
    from parseq_b200.weights import init_state_dict
    m = create_model(experiment, **kw)
    m.model.load_state_dict(init_state_dict(make_config(experiment), seed))
    return m.eval().to("cuda")


def _resize(eng, packed, size):
    out = torch.empty((packed.count, size[0], size[1], 3), dtype=torch.uint8, device="cuda")
    eng.resize_crops(packed, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return out.cpu()


def _pack_cuda(images, rotation):
    from parseq_b200.crops import pack_crops
    return pack_crops([torch.from_numpy(i).cuda() for i in images], rotation)


@pytest.mark.parametrize("size", list(EXPERIMENT_OF_SIZE), ids=lambda s: f"{s[0]}x{s[1]}")
def test_resize_kernel_equals_goldens_and_oracle(size):
    golden = torch.load(GOLDEN, weights_only=False)
    cases = R.golden_crops()
    eng = _model(EXPERIMENT_OF_SIZE[size]).model.engine()
    for rot in R.ROTATIONS:
        idx = [i for i, c in enumerate(cases) if c["rotation"] == rot]
        out = _resize(eng, _pack_cuda([cases[i]["image"] for i in idx], rot), size)
        for k, i in enumerate(idx):
            got = out[k].numpy()
            assert R.digest(got) == golden["outputs"][size][i], (cases[i]["name"], size)
    # oracle recomputed on fresh seeded crops (every size class, each rotation, random and smooth content)
    rng = np.random.default_rng(5)
    fresh = [R._content(rng, h, w, bool(j % 2)) for j, (h, w) in enumerate(
        [(1, 1), (32, 128), (32, 77), (61, 128), (8, 20), (200, 900), (48, 60), (20, 600), (1600, 9), (16, 4096), (33, 129)])]
    for rot in R.ROTATIONS:
        out = _resize(eng, _pack_cuda(fresh, rot), size)
        for k, img in enumerate(fresh):
            assert np.array_equal(out[k].numpy(), R.transform(img, size, rot)), (img.shape, rot, size)


def test_zero_copy_views_equal_packed_copies():
    """Crops that are views into one 1080 x 1920 frame (row stride > 3 * width) are read in place."""
    from parseq_b200.crops import pack_crops
    eng = _model("parseq").model.engine()
    g = torch.Generator().manual_seed(3)
    frame = torch.randint(0, 256, (1080, 1920, 3), dtype=torch.uint8, generator=g).cuda()
    boxes = [(0, 0, 40, 300), (500, 1000, 120, 80), (1079, 1919, 1, 1), (17, 3, 33, 1700), (200, 1900, 700, 20)]
    views = [frame[y:y + h, x:x + w] for y, x, h, w in boxes]
    p_view = pack_crops(views, 90)
    assert p_view.pixels_ptr == frame.data_ptr() and p_view.desc[1].row_stride == 1920 * 3
    p_copy = pack_crops([v.contiguous().clone() for v in views], 90)
    assert p_copy.pixels_ptr != frame.data_ptr()
    a, b = _resize(eng, p_view, (32, 128)), _resize(eng, p_copy, (32, 128))
    assert torch.equal(a, b)
    for k, v in enumerate(views):
        assert np.array_equal(a[k].numpy(), R.transform(v.cpu().numpy(), (32, 128), 90))


def _crops(n, seed):
    """Detector-like crop sizes (heights 12..120, widths 30..900)."""
    rng = np.random.default_rng(seed)
    return [rng.integers(0, 256, (int(rng.integers(12, 121)), int(rng.integers(30, 901)), 3), dtype=np.uint8)
            for _ in range(n)]


def _resized_stack(crops, size, rotation=0):
    return torch.from_numpy(np.stack([R.transform(c, size, rotation) for c in crops]))


@pytest.mark.parametrize("B, decode_ar, refine_iters, max_length", [
    (1, True, 1, None), (7, True, 1, None), (7, False, 2, None), (7, True, 0, None), (7, True, 1, 5),
    (512, True, 1, None), (1000, True, 1, None)])
def test_forward_crops_bit_identical_to_forward_u8(B, decode_ar, refine_iters, max_length):
    """Device and host crop entry points == parseq_forward_u8 on the oracle-resized stack (graph replay; bs 512: fused
    GEMM + LayerNorm and the cluster-of-6 AR regime; bs 1000: two super-chunks; NAR; early exit without refinement)."""
    from parseq_b200.crops import pack_crops
    m = _model("parseq", decode_ar=decode_ar, refine_iters=refine_iters)
    crops = _crops(B, 100 + B)
    rot = 180 if B == 7 else 0
    stack = _resized_stack(crops, (32, 128), rot).cuda()
    with torch.inference_mode():
        ref_l, ref_i = m.model.forward(m.tokenizer, stack, max_length, return_ids=True)
        for packed in (pack_crops([torch.from_numpy(c).cuda() for c in crops], rot), pack_crops(crops, rot)):
            for _ in range(2):                                   # capture, then replay
                lg, ids = m.model.forward_crops(m.tokenizer, packed, max_length, return_ids=True)
                torch.cuda.synchronize()
                assert lg.shape == ref_l.shape and lg.device == ref_l.device
                assert torch.equal(lg, ref_l) and torch.equal(ids, ref_i), packed.host


def test_engine_host_crops_equal_forward_host_u8():
    """parseq_forward_host_crops returns host results equal to parseq_forward_host_u8 on the resized stack, steps too."""
    from parseq_b200.crops import pack_crops
    m = _model("parseq")
    eng = m.model.engine()
    st = torch.cuda.current_stream().cuda_stream
    crops = _crops(300, 7)
    stack = _resized_stack(crops, (32, 128)).pin_memory()
    out = [(torch.empty((300, 26, 95)).pin_memory(), torch.empty((300, 26), dtype=torch.int32).pin_memory(),
            torch.empty((1,), dtype=torch.int32).pin_memory()) for _ in range(2)]
    eng.forward_u8(stack.data_ptr(), 300, *(t.data_ptr() for t in out[0]), st, None, True, 1, host=True)
    eng.forward_crops(pack_crops(crops), *(t.data_ptr() for t in out[1]), st, None, True, 1)
    for a, b in zip(*out):
        assert torch.equal(a, b)


def test_read_equals_postprocess_of_forward_u8():
    m = _model("parseq")
    crops = _crops(9, 11)
    stack = _resized_stack(crops, (32, 128), 90).cuda()
    with torch.inference_mode():
        labels, conf = m.read(crops, rotation=90)
        ref_labels, ref_conf = m.postprocess(m(stack))
    assert labels == ref_labels and conf == ref_conf


def test_vitstr_forward_crops():
    from parseq_b200.crops import pack_crops
    m = _model("vitstr")
    crops = _crops(5, 12)
    stack = _resized_stack(crops, tuple(m.model.cfg.img_size), 270).cuda()
    with torch.inference_mode():
        ref = m(stack)
        assert torch.equal(m.forward_crops(crops, rotation=270), ref)
        assert torch.equal(m.forward_crops(pack_crops([torch.from_numpy(c).cuda() for c in crops], 270)), ref)


def test_invalid_crops_are_rejected_and_the_handle_stays_usable():
    import ctypes as C
    from parseq_b200.crops import pack_crops
    from parseq_b200.engine import CropC, CropsC, ForwardArgsC
    m = _model("parseq")
    eng = m.model.engine()
    lib = eng.lib
    st = torch.cuda.current_stream().cuda_stream
    buf = torch.zeros(64 * 64 * 3, dtype=torch.uint8, device="cuda")
    logits = torch.empty((1, 26, 95), device="cuda")
    out = torch.empty((1, 32, 128, 3), dtype=torch.uint8, device="cuda")
    args = ForwardArgsC(1, -1, 1, 1, None, None)

    def call(crop, rotation=0, resize=False):
        desc = (CropC * 1)(crop)
        cs = CropsC(1, C.cast(desc, C.POINTER(CropC)), buf.data_ptr(), buf.numel(), rotation)
        if resize:
            return lib.parseq_resize_crops(eng.handle, C.byref(cs), out.data_ptr(), st)
        return lib.parseq_forward_crops(eng.handle, C.byref(args), C.byref(cs), logits.data_ptr(), None, None, st)

    ok = CropC(0, 64, 64, 192, 0)
    for resize in (False, True):
        assert call(CropC(64 * 64 * 3 - 10, 8, 8, 24, 0), resize=resize) == -1           # out of bounds
        assert call(CropC(0, 0, 8, 24, 0), resize=resize) == -1                          # zero side
        assert call(CropC(0, 4097, 1, 3, 0), resize=resize) == -1                        # side > 4096
        assert call(ok, rotation=45, resize=resize) == -1                                 # bad rotation
        assert call(ok, resize=resize) == 0                                               # the handle still works
    torch.cuda.synchronize()
    crops = [np.full((64, 64, 3), 77, np.uint8)]
    with torch.inference_mode():
        assert torch.equal(m.model.forward_crops(m.tokenizer, pack_crops([buf.view(64, 64, 3)])),
                           m.model.forward(m.tokenizer, _resized_stack([np.zeros((64, 64, 3), np.uint8)], (32, 128)).cuda()))
        assert torch.equal(m.forward_crops(crops), m(_resized_stack(crops, (32, 128)).cuda()))
