"""Variable-size crop input: cost of the GPU resize and of the whole crop path, against the status quo (PIL resize of
every crop on the host, then parseq_forward_host_u8).  Seeded, detector-like crops: heights 12..120, widths 30..900,
plus a few 1..4 k px extremes.  Prints one JSON line.

    python tests/bench_crops.py [--batch 512] [--iters 20]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def detector_crops(n, seed=0):
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        if i % 64 == 63:                                            # extremes: long lines, tall narrow boxes
            h, w = [(40, 4000), (3000, 40), (1024, 1024)][(i // 64) % 3]
        else:
            h, w = int(rng.integers(12, 121)), int(rng.integers(30, 901))
        out.append(rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    from PIL import Image
    from parseq_b200.config import make_config
    from parseq_b200.crops import pack_crops
    from parseq_b200.factory import create_model
    from parseq_b200.weights import init_state_dict

    B, it = args.batch, args.iters
    m = create_model("parseq")
    m.model.load_state_dict(init_state_dict(make_config("parseq"), 0))
    m = m.eval().to("cuda")
    eng = m.model.engine()
    st = torch.cuda.current_stream().cuda_stream
    crops = detector_crops(B)
    raw_bytes = sum(c.nbytes for c in crops)
    host = pack_crops(crops)
    dev = pack_crops([torch.from_numpy(c).cuda() for c in crops])
    out_u8 = torch.empty((B, 32, 128, 3), dtype=torch.uint8, device="cuda")
    hl = torch.empty((B, 26, 95)).pin_memory()
    hi = torch.empty((B, 26), dtype=torch.int32).pin_memory()
    hs = torch.empty((1,), dtype=torch.int32).pin_memory()

    # resize kernel alone (CUDA events around `it` launches)
    for _ in range(3):
        eng.resize_crops(dev, out_u8.data_ptr(), st)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(it):
        eng.resize_crops(dev, out_u8.data_ptr(), st)
    b.record()
    torch.cuda.synchronize()
    resize_us = a.elapsed_time(b) * 1e3 / it

    def wall(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(it):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) / it

    t_crops = wall(lambda: eng.forward_crops(host, hl.data_ptr(), hi.data_ptr(), hs.data_ptr(), st))

    def status_quo():
        stack = np.stack([np.asarray(Image.fromarray(c).resize((128, 32), Image.BICUBIC)) for c in crops])
        pinned = torch.from_numpy(stack).pin_memory()
        eng.forward_u8(pinned.data_ptr(), B, hl.data_ptr(), hi.data_ptr(), hs.data_ptr(), st, None, True, 1, host=True)
    t_quo = wall(status_quo)

    dev_name = torch.cuda.get_device_name(0)
    print(json.dumps(dict(
        device=dev_name, batch=B, iters=it,
        resize_kernel_us_per_batch=round(resize_us, 1),
        forward_host_crops_ms=round(t_crops * 1e3, 3), forward_host_crops_per_s=round(B / t_crops, 1),
        pil_resize_plus_forward_host_u8_ms=round(t_quo * 1e3, 3), pil_resize_plus_forward_host_u8_per_s=round(B / t_quo, 1),
        h2d_bytes_crops=int(host.pixels_bytes), h2d_bytes_resized=B * 32 * 128 * 3, raw_crop_bytes=int(raw_bytes))))


if __name__ == "__main__":
    main()
