"""Imports the reference's own `strhub.models.parseq.model.PARSeq` from the reference tree (REF_ROOT, read-only)
under the timm shim.  TEST INFRASTRUCTURE ONLY: used by oracle/make_golden.py, which stores the reference's outputs
under tests/golden; the tests compare against those and never import the reference.

Where the reference tree is absent, the byte-compiled copy `oracle/_ref/` (oracle/build_ref.py) is imported instead,
and only by bench.py's CPU legs (`--impl reference`, `cpu_baseline`).
"""
from __future__ import annotations

import importlib
import os
import sys

REF_ROOT = os.environ.get("PARSEQ_REFERENCE_ROOT", "/root/reference")
# byte-compiled copy of the same modules made by oracle/build_ref.py (travels to the GPU box; binaries only)
_REF_PYC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
if not os.path.isfile(os.path.join(REF_ROOT, "strhub/models/parseq/model.py")) and \
        os.path.isfile(os.path.join(_REF_PYC, "strhub/models/parseq/model.pyc")):
    REF_ROOT = _REF_PYC


def available() -> bool:
    return os.path.isfile(os.path.join(REF_ROOT, "strhub/models/parseq/model.py")) or \
        os.path.isfile(os.path.join(REF_ROOT, "strhub/models/parseq/model.pyc"))


def kind() -> str:
    """'source' (the reference tree itself), 'pyc' (oracle/_ref, byte-compiled from it) or 'absent'."""
    if os.path.isfile(os.path.join(REF_ROOT, "strhub/models/parseq/model.py")):
        return "source"
    return "pyc" if available() else "absent"


def load_reference_classes():
    """Returns (RefPARSeqModel, RefTokenizer) imported from the reference tree.

    The repo root also has a `strhub` package (the drop-in boundary); to import the REFERENCE one
    its modules are loaded under the private alias `_refstrhub` by temporarily swapping sys.modules.
    """
    from . import timm_shim
    timm_shim.install()
    saved = {k: v for k, v in sys.modules.items() if k == "strhub" or k.startswith("strhub.")}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, REF_ROOT)
    try:
        model_mod = importlib.import_module("strhub.models.parseq.model")
        data_mod = importlib.import_module("strhub.data.utils")
        assert os.path.realpath(model_mod.__file__).startswith(os.path.realpath(REF_ROOT)), model_mod.__file__
        Ref, Tok = model_mod.PARSeq, data_mod.Tokenizer
    finally:
        sys.path.remove(REF_ROOT)
        for k in [k for k in sys.modules if k == "strhub" or k.startswith("strhub.")]:
            del sys.modules[k]
        sys.modules.update(saved)
    return Ref, Tok


def load_reference_vitstr_class():
    """The reference's inner `strhub.models.vitstr.model.ViTSTR` (a timm VisionTransformer subclass; under the shim).
    The Lightning system around it (vitstr/system.py) needs pytorch_lightning / nltk and is restated by
    oracle/vitstr_oracle.py:system_forward instead."""
    from . import timm_shim
    timm_shim.install()
    saved = {k: v for k, v in sys.modules.items() if k == "strhub" or k.startswith("strhub.")}
    for k in saved:
        del sys.modules[k]
    import types
    sys.path.insert(0, REF_ROOT)
    try:
        # bypass strhub/models/vitstr/__init__ -> system.py (pytorch_lightning): load model.py as a plain module
        for pkg in ("strhub", "strhub.models", "strhub.models.vitstr"):
            m = types.ModuleType(pkg)
            m.__path__ = [os.path.join(REF_ROOT, *pkg.split("."))]
            sys.modules[pkg] = m
        mod = importlib.import_module("strhub.models.vitstr.model")
        assert os.path.realpath(mod.__file__).startswith(os.path.realpath(REF_ROOT)), mod.__file__
        cls = mod.ViTSTR
    finally:
        sys.path.remove(REF_ROOT)
        for k in [k for k in sys.modules if k == "strhub" or k.startswith("strhub.")]:
            del sys.modules[k]
        sys.modules.update(saved)
    return cls


def build_reference_vitstr(cfg, state_dict):
    """ctor arguments of vitstr/system.py:50-59."""
    cls = load_reference_vitstr_class()
    m = cls(img_size=list(cfg.img_size), patch_size=list(cfg.patch_size), depth=cfg.enc_depth, mlp_ratio=cfg.enc_mlp_ratio,
            qkv_bias=True, embed_dim=cfg.embed_dim, num_heads=cfg.enc_num_heads, num_classes=cfg.num_classes)
    m.load_state_dict(state_dict, strict=True)
    return m.eval()


def build_reference_model(cfg, state_dict):
    Ref, Tok = load_reference_classes()
    tok = Tok(cfg.charset_train)
    m = Ref(len(tok), cfg.max_label_length, list(cfg.img_size), list(cfg.patch_size), cfg.embed_dim,
            cfg.enc_num_heads, cfg.enc_mlp_ratio, cfg.enc_depth, cfg.dec_num_heads, cfg.dec_mlp_ratio,
            cfg.dec_depth, cfg.decode_ar, cfg.refine_iters, cfg.dropout)
    missing, unexpected = m.load_state_dict(state_dict, strict=True), None
    return m.eval(), tok
