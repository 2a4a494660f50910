"""ctypes binding of include/parseq_b200.h.  The library is the product; this file only marshals
pointers.  There is no fallback: if the shared library is missing or no sm_100 device exists,
construction raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional

from .build import LIB_PATH

_lib = None


class ParseqConfigC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "img_h", "img_w", "patch_h", "patch_w", "embed_dim", "enc_num_heads", "enc_mlp_ratio", "enc_depth",
        "dec_num_heads", "dec_mlp_ratio", "dec_depth", "max_label_length", "num_tokens", "max_batch", "device", "arch")]


class ForwardArgsC(C.Structure):
    _fields_ = [("batch", C.c_int32), ("max_length", C.c_int32), ("decode_ar", C.c_int32),
                ("refine_iters", C.c_int32), ("forced_ids", C.c_void_p), ("forced_refine", C.c_void_p)]


class CropC(C.Structure):
    _fields_ = [("offset", C.c_int64), ("height", C.c_int32), ("width", C.c_int32), ("row_stride", C.c_int32),
                ("reserved", C.c_int32)]


class CropsC(C.Structure):
    _fields_ = [("count", C.c_int32), ("desc", C.POINTER(CropC)), ("pixels", C.c_void_p), ("pixels_bytes", C.c_int64),
                ("rotation", C.c_int32)]


EXPORTS = [
    "parseq_create", "parseq_destroy", "parseq_set_weight", "parseq_num_weights", "parseq_weight_key",
    "parseq_finalize", "parseq_forward", "parseq_forward_host", "parseq_forward_u8", "parseq_forward_host_u8",
    "parseq_postprocess", "parseq_encode", "parseq_decode", "parseq_head", "parseq_text_embed", "parseq_kernel_launches", "parseq_debug_int", "parseq_bench_tma_stream",
    "parseq_set_option", "parseq_get_timing", "parseq_get_ar_profile", "parseq_last_error", "parseq_version", "parseq_gemm_bf16", "parseq_gemm_ln_bf16", "parseq_mlp_ln_bf16", "parseq_mlp_ln_bf16_prof", "parseq_layernorm_bf16",
    "parseq_enc_attention", "parseq_forward_crops", "parseq_forward_host_crops", "parseq_resize_crops",
]


def load_library(path: Optional[str] = None):
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("PARSEQ_B200_LIB", LIB_PATH)
    if not os.path.exists(p):
        raise RuntimeError(f"{p} not found: build it with `python -m parseq_b200.build` "
                           "(there is no CPU / PyTorch fallback)")
    lib = C.CDLL(p)
    lib.parseq_last_error.restype = C.c_char_p
    lib.parseq_version.restype = C.c_char_p
    lib.parseq_weight_key.restype = C.c_char_p
    lib.parseq_weight_key.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int64)]
    lib.parseq_bench_tma_stream.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    lib.parseq_debug_int.restype = C.c_int64
    lib.parseq_debug_int.argtypes = [C.c_void_p, C.c_char_p]
    lib.parseq_kernel_launches.restype = C.c_int64
    lib.parseq_kernel_launches.argtypes = [C.c_void_p]
    lib.parseq_create.argtypes = [C.POINTER(ParseqConfigC), C.POINTER(C.c_void_p)]
    lib.parseq_destroy.argtypes = [C.c_void_p]
    lib.parseq_destroy.restype = None
    lib.parseq_set_weight.argtypes = [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]
    lib.parseq_num_weights.argtypes = [C.c_void_p]
    lib.parseq_finalize.argtypes = [C.c_void_p, C.c_void_p]
    lib.parseq_forward.argtypes = [C.c_void_p, C.POINTER(ForwardArgsC), C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p]
    lib.parseq_forward_host.argtypes = lib.parseq_forward.argtypes
    lib.parseq_forward_u8.argtypes = lib.parseq_forward.argtypes
    lib.parseq_forward_host_u8.argtypes = lib.parseq_forward.argtypes
    lib.parseq_forward_crops.argtypes = [C.c_void_p, C.POINTER(ForwardArgsC), C.POINTER(CropsC), C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]
    lib.parseq_forward_host_crops.argtypes = lib.parseq_forward_crops.argtypes
    lib.parseq_resize_crops.argtypes = [C.c_void_p, C.POINTER(CropsC), C.c_void_p, C.c_void_p]
    lib.parseq_postprocess.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]
    lib.parseq_encode.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.parseq_decode.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p]
    lib.parseq_head.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.parseq_text_embed.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.parseq_set_option.argtypes = [C.c_void_p, C.c_char_p, C.c_int64]
    lib.parseq_get_timing.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                      C.POINTER(C.c_int64)]
    lib.parseq_gemm_bf16.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                                     C.c_int64, C.c_void_p]
    lib.parseq_gemm_ln_bf16.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]
    lib.parseq_mlp_ln_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]
    lib.parseq_mlp_ln_bf16_prof.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.parseq_layernorm_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_int,
                                          C.c_void_p, C.c_void_p, C.c_void_p]
    lib.parseq_enc_attention.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    if path is None:
        _lib = lib
    return lib


class EngineError(RuntimeError):
    pass


def check(lib, rc: int):
    if rc != 0:
        raise EngineError(f"parseq_b200 error {rc}: {lib.parseq_last_error().decode()}")


class Engine:
    """Owns one `parseq_engine*`."""

    def __init__(self, cfg, device: int = 0, max_batch: int = 0):
        self.lib = load_library()
        self.cfg = cfg
        c = ParseqConfigC(cfg.img_size[0], cfg.img_size[1], cfg.patch_size[0], cfg.patch_size[1], cfg.embed_dim,
                          cfg.enc_num_heads, cfg.enc_mlp_ratio, cfg.enc_depth, cfg.dec_num_heads, cfg.dec_mlp_ratio,
                          cfg.dec_depth, cfg.max_label_length, cfg.num_tokens, max_batch, device,
                          1 if getattr(cfg, "arch", "parseq") == "vitstr" else 0)
        h = C.c_void_p()
        check(self.lib, self.lib.parseq_create(C.byref(c), C.byref(h)))
        self.handle = h
        self.device = device

    def close(self):
        if getattr(self, "handle", None):
            self.lib.parseq_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def weight_keys(self) -> Dict[str, int]:
        out = {}
        n = self.lib.parseq_num_weights(self.handle)
        for i in range(n):
            numel = C.c_int64()
            k = self.lib.parseq_weight_key(self.handle, i, C.byref(numel))
            out[k.decode()] = numel.value
        return out

    def load_state_dict(self, sd, stream: int = 0):
        import torch
        expected = self.weight_keys()
        missing = [k for k in expected if k not in sd]
        unexpected = [k for k in sd if k not in expected]
        if missing or unexpected:
            raise EngineError(f"state_dict mismatch: missing {missing[:4]}... unexpected {unexpected[:4]}...")
        for k, numel in expected.items():
            t = sd[k].detach().to(device="cpu", dtype=torch.float32).contiguous()
            if t.numel() != numel:
                raise EngineError(f"size mismatch for {k}: {tuple(t.shape)} vs {numel} elements")
            check(self.lib, self.lib.parseq_set_weight(self.handle, k.encode(), t.data_ptr(), numel))
        check(self.lib, self.lib.parseq_finalize(self.handle, stream))

    def set_option(self, name: str, value: int):
        check(self.lib, self.lib.parseq_set_option(self.handle, name.encode(), int(value)))

    TIMING_CATEGORIES = ("enc_gemm", "enc_attn", "layernorm", "dec_gemm", "dec_attn", "other", "enc_gemm_ln", "dec_ar")

    def get_timing(self):
        out = {}
        for i, name in enumerate(self.TIMING_CATEGORIES):
            ms, fl, n = C.c_double(), C.c_double(), C.c_int64()
            check(self.lib, self.lib.parseq_get_timing(self.handle, i, C.byref(ms), C.byref(fl), C.byref(n)))
            out[name] = dict(ms=ms.value, flops=fl.value, launches=n.value)
        return out

    def get_ar_profile(self):
        buf = (C.c_uint64 * 512)()
        self.lib.parseq_get_ar_profile.argtypes = [C.c_void_p, C.POINTER(C.c_uint64)]
        check(self.lib, self.lib.parseq_get_ar_profile(self.handle, buf))
        return [[buf[s * 16 + k] for k in range(16)] for s in range(32)]

    def debug_int(self, name: str) -> int:
        return int(self.lib.parseq_debug_int(self.handle, name.encode()))

    @property
    def launches(self) -> int:
        return int(self.lib.parseq_kernel_launches(self.handle))

    def num_steps(self, max_length) -> int:
        ml = self.cfg.max_label_length if max_length is None else min(int(max_length), self.cfg.max_label_length)
        return ml + 1

    def _args(self, batch, max_length, decode_ar, refine_iters, forced_ids=None, forced_refine=None):
        return ForwardArgsC(batch, -1 if max_length is None else int(max_length), int(bool(decode_ar)),
                            int(refine_iters), forced_ids, forced_refine)

    def forward(self, images_ptr, batch, logits_ptr, ids_ptr, steps_ptr, stream, max_length=None, decode_ar=True,
                refine_iters=1, forced_ids_ptr=None, forced_refine_ptr=None):
        a = self._args(batch, max_length, decode_ar, refine_iters, forced_ids_ptr, forced_refine_ptr)
        check(self.lib, self.lib.parseq_forward(self.handle, C.byref(a), images_ptr, logits_ptr, ids_ptr, steps_ptr,
                                                stream))

    def forward_host(self, images_ptr, batch, logits_ptr, ids_ptr, steps_ptr, stream, max_length=None,
                     decode_ar=True, refine_iters=1):
        a = self._args(batch, max_length, decode_ar, refine_iters)
        check(self.lib, self.lib.parseq_forward_host(self.handle, C.byref(a), images_ptr, logits_ptr, ids_ptr,
                                                     steps_ptr, stream))

    def forward_u8(self, images_ptr, batch, logits_ptr, ids_ptr, steps_ptr, stream, max_length=None, decode_ar=True,
                   refine_iters=1, host=False):
        a = self._args(batch, max_length, decode_ar, refine_iters)
        fn = self.lib.parseq_forward_host_u8 if host else self.lib.parseq_forward_u8
        check(self.lib, fn(self.handle, C.byref(a), images_ptr, logits_ptr, ids_ptr, steps_ptr, stream))

    def forward_crops(self, crops, logits_ptr, ids_ptr, steps_ptr, stream, max_length=None, decode_ar=True,
                      refine_iters=1):
        """`crops`: a `parseq_b200.crops.PackedCrops`; host pixels run parseq_forward_host_crops (host outputs,
        synchronised on return), device pixels parseq_forward_crops (device outputs, enqueued on `stream`)."""
        a = self._args(crops.count, max_length, decode_ar, refine_iters)
        fn = self.lib.parseq_forward_host_crops if crops.host else self.lib.parseq_forward_crops
        check(self.lib, fn(self.handle, C.byref(a), C.byref(crops.c_struct()), logits_ptr, ids_ptr, steps_ptr, stream))

    def resize_crops(self, crops, out_ptr, stream):
        """Device crops -> uint8 [count, img_h, img_w, 3] at `out_ptr` (device)."""
        check(self.lib, self.lib.parseq_resize_crops(self.handle, C.byref(crops.c_struct()), out_ptr, stream))

    def postprocess(self, logits_ptr, batch, num_steps, ids_ptr, lengths_ptr, conf_ptr, stream, eos_id=0):
        check(self.lib, self.lib.parseq_postprocess(logits_ptr, batch, num_steps, self.cfg.num_classes, eos_id, ids_ptr,
                                                    lengths_ptr, conf_ptr, stream))

    def encode(self, images_ptr, batch, memory_ptr, stream):
        check(self.lib, self.lib.parseq_encode(self.handle, batch, images_ptr, memory_ptr, stream))

    def decode(self, batch, ctx_len, num_queries, tgt_ptr, memory_ptr, query_ptr, qmask_ptr, pmask_ptr, out_ptr, stream):
        check(self.lib, self.lib.parseq_decode(self.handle, batch, ctx_len, num_queries, tgt_ptr, memory_ptr, query_ptr,
                                               qmask_ptr, pmask_ptr, out_ptr, stream))

    def head(self, rows, x_ptr, logits_ptr, stream):
        check(self.lib, self.lib.parseq_head(self.handle, rows, x_ptr, logits_ptr, stream))

    def text_embed(self, n, ids_ptr, out_ptr, stream):
        check(self.lib, self.lib.parseq_text_embed(self.handle, n, ids_ptr, out_ptr, stream))
