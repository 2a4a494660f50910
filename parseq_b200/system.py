"""Drop-in Python surface of the PARSeq inference path.

`PARSeq` mirrors `strhub.models.parseq.system.PARSeq` (system.py:33-88: ctor kwargs, `.model`,
`.tokenizer`, `.hparams`, `forward(images, max_length)`) and the bits of `BaseSystem` its callers use
(`test_step` -> `BatchResult`, base.py:36-44,112-143,179-180; `.device`).  `ParseqModel` mirrors the
inner `strhub.models.parseq.model.PARSeq` (model.py:31-169): same parameter names (so released
`parseq-*.pt` state_dicts load), `encode`, `forward(tokenizer, images, max_length)`, `decode_ar`,
`refine_iters`, `max_label_length`.  All arithmetic happens in libparseq_b200.so (sm_100a CUDA);
these classes only own the parameters and marshal pointers.  There is no CPU or eager-PyTorch
fallback: calling forward with non-CUDA tensors raises.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from types import SimpleNamespace
from typing import Any, Dict, Optional, Sequence

import torch
from torch import Tensor, nn

from .config import ParseqConfig, make_config
from .engine import Engine, EngineError
from .tokenizer import CharsetAdapter, Tokenizer


class InvalidModelError(RuntimeError):
    """Raised for any model-related error (creation, loading) — name kept from strhub/models/utils.py:10."""


@dataclass
class BatchResult:          # base.py:36-44
    num_samples: int
    correct: int
    ned: float
    confidence: float
    label_length: int
    loss: Optional[Tensor]
    loss_numel: Optional[int]


def edit_distance(a: str, b: str) -> int:
    """Levenshtein distance (the reference uses nltk.edit_distance, base.py:29,139)."""
    if a == b:
        return 0
    if not a or not b:
        return len(a) + len(b)
    prev = list(range(len(b) + 1))
    for i, ca in enumerate(a, 1):
        cur = [i]
        for j, cb in enumerate(b, 1):
            cur.append(min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (ca != cb)))
        prev = cur
    return prev[-1]


class _Holder(nn.Module):
    """Parameter container; nested so that state_dict keys equal the reference's."""


class _HeadModule(_Holder):
    """`model.head` (model.py:63, nn.Linear(embed_dim, num_tokens - 2)) as a callable: x [..., D] fp32 -> logits."""

    def forward(self, x: Tensor) -> Tensor:
        owner = self.__dict__["_owner"]()
        eng = owner.engine()
        D = owner.cfg.embed_dim
        if x.device.type != "cuda":
            raise RuntimeError("head() takes CUDA tensors (no CPU fallback)")
        x2 = x.to(torch.float32).reshape(-1, D).contiguous()
        out = torch.empty((x2.shape[0], owner.cfg.num_classes), dtype=torch.float32, device=x.device)
        eng.head(x2.shape[0], x2.data_ptr(), out.data_ptr(), torch.cuda.current_stream(x.device).cuda_stream)
        return out.reshape(*x.shape[:-1], owner.cfg.num_classes)


class _TextEmbedModule(_Holder):
    """`model.text_embed` (modules.py:168-176, TokenEmbedding) as a callable: ids [...] -> sqrt(D) * embedding[ids]."""

    def forward(self, tokens: Tensor) -> Tensor:
        owner = self.__dict__["_owner"]()
        eng = owner.engine()
        if tokens.device.type != "cuda":
            raise RuntimeError("text_embed() takes CUDA tensors (no CPU fallback)")
        ids = tokens.to(torch.int32).contiguous()
        out = torch.empty((*ids.shape, owner.cfg.embed_dim), dtype=torch.float32, device=ids.device)
        eng.text_embed(ids.numel(), ids.data_ptr(), out.data_ptr(), torch.cuda.current_stream(ids.device).cuda_stream)
        return out


def _register(root: nn.Module, key: str, tensor: Tensor):
    parts = key.split(".")
    mod = root
    for p in parts[:-1]:
        if not hasattr(mod, p):
            mod.add_module(p, _Holder())
        mod = getattr(mod, p)
    mod.register_parameter(parts[-1], nn.Parameter(tensor, requires_grad=False))


class _EngineModule(nn.Module):
    """Owns the parameters (reference state_dict names) and the lazily created engine handle."""

    def __init__(self, cfg: ParseqConfig):
        super().__init__()
        from .weights import init_state_dict
        self.cfg = cfg
        self.max_label_length = cfg.max_label_length
        # random init with the reference's distributions (weights.py); bf16-exact not forced here
        for k, v in init_state_dict(cfg, seed=0, perturb=False, bf16_exact=False).items():
            _register(self, k, v)
        self._engine: Optional[Engine] = None
        self._engine_sig = None
        self._options = {}
        # `head` / `text_embed` are callable like the reference's submodules (they hold the same parameters)
        import weakref
        for name, cls in (("head", _HeadModule), ("text_embed", _TextEmbedModule)):
            if hasattr(self, name):
                mod = getattr(self, name)
                mod.__class__ = cls
                mod.__dict__["_owner"] = weakref.ref(self)

    # ---- engine plumbing -------------------------------------------------------------------
    @property
    def _device(self) -> torch.device:
        return next(self.parameters()).device

    def _signature(self):
        """Cheap staleness check of the engine's weight copy: version counters of every parameter (in-place updates,
        load_state_dict) + the storage addresses of the first / last one (`.to()` moves).  The parameter list is cached:
        walking the module tree costs more than a bs=1 forward's launch overhead."""
        pl = self.__dict__.get("_plist")
        if pl is None:
            pl = list(self.parameters())
            self.__dict__["_plist"] = pl
        try:
            vers = tuple(p._version for p in pl)
        except RuntimeError:           # inference tensors carry no version counter
            vers = tuple(id(p) for p in pl)
        return (vers, pl[0].data_ptr(), pl[-1].data_ptr(), len(pl))

    def _apply(self, fn, *args, **kwargs):
        out = super()._apply(fn, *args, **kwargs)
        self.__dict__.pop("_plist", None)
        self._engine_sig = None
        return out

    def engine(self) -> Engine:
        dev = self._device
        if dev.type != "cuda":
            raise RuntimeError("parseq_b200 runs on a CUDA (sm_100a) device only; move the model with .to('cuda') "
                               "— there is no CPU fallback")
        idx = dev.index if dev.index is not None else torch.cuda.current_device()
        if self._engine is None or self._engine.device != idx:
            self._engine = Engine(self.cfg, idx)
            for name, value in self._options.items():
                self._engine.set_option(name, value)
            self._engine_sig = None
        sig = self._signature()
        if sig != self._engine_sig:
            self._engine.load_state_dict(self.state_dict(), torch.cuda.current_stream(idx).cuda_stream)
            self._engine_sig = sig
        return self._engine

    def set_engine_option(self, name: str, value: int):
        """Engine tuning knobs: "max_batch", "chunk", "use_graph" (see include/parseq_b200.h)."""
        self._options[name] = int(value)
        if self._engine is not None:
            self._engine.set_option(name, value)

    def _check_images(self, images: Tensor) -> Tensor:
        if images.device.type != "cuda":
            raise RuntimeError("images must be CUDA tensors (no CPU fallback)")
        H, W = self.cfg.img_size
        if images.dtype == torch.uint8:      # raw crops [N, H, W, 3]: ToTensor + Normalize(0.5, 0.5) run inside the engine
            if images.dim() != 4 or tuple(images.shape[1:]) != (H, W, 3):
                raise AssertionError(f"uint8 input must be (N,{H},{W},3), got {tuple(images.shape)}")
            return images.contiguous()
        if images.dim() != 4 or images.shape[1] != 3 or tuple(images.shape[-2:]) != (H, W):
            raise AssertionError(f"Input image size {tuple(images.shape)} doesn't match model (N,3,{H},{W})")
        return images.to(torch.float32).contiguous()

    def _features(self, img: Tensor) -> Tensor:
        """timm forward_features of the ViT: fp32 [N, tokens, D]."""
        eng = self.engine()
        img = self._check_images(img)
        if img.dtype == torch.uint8:
            raise AssertionError("encode / forward_features take normalised float images")
        mem = torch.empty((img.shape[0], self.cfg.enc_tokens, self.cfg.embed_dim), dtype=torch.float32,
                          device=img.device)
        eng.encode(img.data_ptr(), img.shape[0], mem.data_ptr(), torch.cuda.current_stream(img.device).cuda_stream)
        return mem

    def _run(self, images: Tensor, max_length, decode_ar, refine_iters, forced_ids=None, forced_refine=None):
        eng = self.engine()
        images = self._check_images(images)
        dev = images.device
        N = images.shape[0]
        L = eng.num_steps(max_length)
        logits = torch.empty((N, L, self.cfg.num_classes), dtype=torch.float32, device=dev)
        ids = torch.empty((N, L), dtype=torch.int32, device=dev)
        steps = torch.empty((1,), dtype=torch.int32, device=dev)
        fi = forced_ids.to(device=dev, dtype=torch.int32).contiguous() if forced_ids is not None else None
        fr = forced_refine.to(device=dev, dtype=torch.int32).contiguous() if forced_refine is not None else None
        st = torch.cuda.current_stream(dev).cuda_stream
        if images.dtype == torch.uint8:
            eng.forward_u8(images.data_ptr(), N, logits.data_ptr(), ids.data_ptr(), steps.data_ptr(), st, max_length,
                           decode_ar, refine_iters)
        else:
            eng.forward(images.data_ptr(), N, logits.data_ptr(), ids.data_ptr(), steps.data_ptr(), st, max_length,
                        decode_ar, refine_iters, fi.data_ptr() if fi is not None else None,
                        fr.data_ptr() if fr is not None else None)
        return logits, ids, steps

    def _run_crops(self, crops, max_length, decode_ar, refine_iters, rotation):
        """Variable-size RGB crops (see parseq_b200.crops): rotate + bicubic resize + normalise on the GPU, then the
        uint8 path.  Outputs are on the model's device whatever the crops' location."""
        from .crops import PackedCrops, pack_crops
        eng = self.engine()
        packed = crops if isinstance(crops, PackedCrops) else pack_crops(crops, rotation)
        dev = self._device
        N, L = packed.count, eng.num_steps(max_length)
        shapes = ((N, L, self.cfg.num_classes), (N, L), (1,))
        if not packed.host and packed.device != dev:
            raise RuntimeError(f"crops are on {packed.device}, the model on {dev}")
        pin = packed.host
        where = dict(pin_memory=True) if pin else dict(device=dev)
        logits, ids, steps = (torch.empty(shp, dtype=dt, **where)
                              for shp, dt in zip(shapes, (torch.float32, torch.int32, torch.int32)))
        if N == 0:
            steps.fill_(L)
        else:
            eng.forward_crops(packed, logits.data_ptr(), ids.data_ptr(), steps.data_ptr(),
                              torch.cuda.current_stream(dev).cuda_stream, max_length, decode_ar, refine_iters)
        if pin:             # the host entry point returns synchronised host results
            logits, ids, steps = (t.to(dev, non_blocking=True) for t in (logits, ids, steps))
        return logits, ids, steps


class ParseqModel(_EngineModule):
    def __init__(self, cfg: ParseqConfig):
        super().__init__(cfg)
        self.decode_ar = cfg.decode_ar
        self.refine_iters = cfg.refine_iters

    # ---- reference API ---------------------------------------------------------------------
    def encode(self, img: Tensor) -> Tensor:
        return self._features(img)

    @staticmethod
    def _bool_mask(mask: Optional[Tensor], shape, dev) -> Optional[Tensor]:
        """torch's attention masks are bool (True = masked) or additive floats (-inf = masked, 0 = keep)."""
        if mask is None:
            return None
        if mask.dtype == torch.bool:
            m = mask
        elif mask.is_floating_point():
            if bool(((mask != 0) & ~torch.isneginf(mask)).any()):
                raise NotImplementedError("additive attention masks other than 0 / -inf are not supported by the engine")
            m = torch.isneginf(mask)
        else:
            m = mask != 0
        if tuple(m.shape) != tuple(shape):
            raise AssertionError(f"mask shape {tuple(m.shape)} != {tuple(shape)}")
        return m.to(device=dev, dtype=torch.uint8).contiguous()

    def decode(self, tgt: Tensor, memory: Tensor, tgt_mask: Optional[Tensor] = None,
               tgt_padding_mask: Optional[Tensor] = None, tgt_query: Optional[Tensor] = None,
               tgt_query_mask: Optional[Tensor] = None) -> Tensor:
        """model.py:86-103: decoder output [N, NQ, D] (before `head`) for context ids `tgt` [N, J] and encoder `memory`
        [N, T, D].  `tgt_mask` acts on the content stream only, which the depth-1 decoder never updates
        (modules.py:117-123), so it is accepted and ignored."""
        eng = self.engine()
        dev = memory.device
        if dev.type != "cuda" or tgt.device != dev:
            raise RuntimeError("decode() takes CUDA tensors (no CPU fallback)")
        N, J = tgt.shape
        D, T = self.cfg.embed_dim, self.cfg.enc_tokens
        if tuple(memory.shape) != (N, T, D):
            raise AssertionError(f"memory shape {tuple(memory.shape)} != {(N, T, D)}")
        ids = tgt.to(torch.int32).contiguous()
        mem = memory.to(torch.float32).contiguous()
        q = None
        NQ = J
        if tgt_query is not None:
            NQ = tgt_query.shape[1]
            q = tgt_query.to(device=dev, dtype=torch.float32).expand(N, NQ, D).contiguous()
        qm = self._bool_mask(tgt_query_mask, (NQ, J), dev)
        pm = self._bool_mask(tgt_padding_mask, (N, J), dev)
        out = torch.empty((N, NQ, D), dtype=torch.float32, device=dev)
        eng.decode(N, J, NQ, ids.data_ptr(), mem.data_ptr(), q.data_ptr() if q is not None else None,
                   qm.data_ptr() if qm is not None else None, pm.data_ptr() if pm is not None else None, out.data_ptr(),
                   torch.cuda.current_stream(dev).cuda_stream)
        return out

    def forward(self, tokenizer: Tokenizer, images: Tensor, max_length: Optional[int] = None,
                return_ids: bool = False, forced_ids: Optional[Tensor] = None,
                forced_refine: Optional[Tensor] = None):
        logits, ids, steps = self._run(images, max_length, self.decode_ar, self.refine_iters, forced_ids, forced_refine)
        return self._finish(logits, ids, steps, max_length, return_ids)

    def forward_crops(self, tokenizer: Tokenizer, crops, max_length: Optional[int] = None, rotation: int = 0,
                      return_ids: bool = False):
        """`forward` on variable-size RGB crops (PIL images, uint8 numpy / torch [h, w, 3], or a PackedCrops) with the
        reference's input transform - rotate(rotation, expand=True), Resize(img_size, BICUBIC), ToTensor, Normalize -
        run on the GPU; bit-identical to `forward` on the uint8 stack PIL's resize produces."""
        logits, ids, steps = self._run_crops(crops, max_length, self.decode_ar, self.refine_iters, rotation)
        return self._finish(logits, ids, steps, max_length, return_ids)

    def _finish(self, logits, ids, steps, max_length, return_ids):
        if max_length is None and self.decode_ar and not self.refine_iters:
            # model.py:144-147: with no refinement the reference returns only the S steps it ran
            S = int(steps.item())
            logits, ids = logits[:, :S], ids[:, :S]
        if return_ids:
            return logits, ids
        return logits


class VitstrModel(_EngineModule):
    """Mirror of `strhub.models.vitstr.model.ViTSTR` (vitstr/model.py:14-28): a timm ViT with class token whose head is
    applied per token.  Parameters carry timm's names (`cls_token`, `pos_embed`, `blocks.<i>...`, `norm`, `head`)."""

    def forward_features(self, x: Tensor) -> Tensor:
        return self._features(x)

    def forward_tokens(self, images: Tensor, max_length: Optional[int] = None, return_ids: bool = False):
        """`self.forward(images, max_length + 2)[:, 1:]` (vitstr/system.py:65-71) in one engine call."""
        logits, ids, _ = self._run(images, max_length, False, 0)
        return (logits, ids) if return_ids else logits

    def forward_tokens_crops(self, crops, max_length: Optional[int] = None, rotation: int = 0, return_ids: bool = False):
        """`forward_tokens` on variable-size RGB crops (see ParseqModel.forward_crops)."""
        logits, ids, _ = self._run_crops(crops, max_length, False, 0, rotation)
        return (logits, ids) if return_ids else logits

    def forward(self, x: Tensor, seqlen: int = 25) -> Tensor:
        raise NotImplementedError(
            "the engine computes head(norm(x))[:, 1:seqlen] only: token 0 (the class token) is discarded by the only "
            "reference caller (vitstr/system.py:68-70); use forward_tokens(images, max_length) or forward_features(x)")


class _HParams(SimpleNamespace):
    def __getitem__(self, k):
        return getattr(self, k)

    def __contains__(self, k):
        return hasattr(self, k)

    def keys(self):
        return self.__dict__.keys()


class _System(nn.Module):
    """The inference-side surface of `strhub.models.base.CrossEntropySystem` (base.py:36-44,112-143,179-207)."""

    def _init_base(self, charset_train, charset_test, batch_size, lr, warmup_pct, weight_decay):
        self.tokenizer = Tokenizer(charset_train)
        self.charset_adapter = CharsetAdapter(charset_test)
        self.bos_id, self.eos_id, self.pad_id = self.tokenizer.bos_id, self.tokenizer.eos_id, self.tokenizer.pad_id
        self.batch_size, self.lr, self.warmup_pct, self.weight_decay = batch_size, lr, warmup_pct, weight_decay

    @property
    def device(self) -> torch.device:
        return self.model._device

    def postprocess(self, logits: Tensor):
        """Device-side greedy decode of logits [N, L, C]: (labels, confidences) with the semantics of
        `logits.softmax(-1)` -> `tokenizer.decode` -> `prob.prod()` (base.py:132-142); one small D2H per batch."""
        eng = self.model.engine()
        logits = logits.contiguous()
        N, L, _ = logits.shape
        dev = logits.device
        ids = torch.empty((N, L), dtype=torch.int32, device=dev)
        lengths = torch.empty((N,), dtype=torch.int32, device=dev)
        conf = torch.empty((N,), dtype=torch.float32, device=dev)
        eng.postprocess(logits.data_ptr(), N, L, ids.data_ptr(), lengths.data_ptr(), conf.data_ptr(),
                        torch.cuda.current_stream(dev).cuda_stream, self.eos_id)
        ids_h, len_h, conf_h = ids.cpu().tolist(), lengths.cpu().tolist(), conf.cpu().tolist()
        labels = [self.tokenizer._ids2tok(row[:n], True) for row, n in zip(ids_h, len_h)]
        return labels, conf_h

    def read(self, crops, rotation: int = 0):
        """The reference's read.py in one call: variable-size RGB crops -> (labels, confidences)."""
        return self.postprocess(self.forward_crops(crops, rotation=rotation))

    # base.py:112-143,179-180 (test path only; validation loss is a training concern)
    def _eval_step(self, batch, validation: bool = False):
        images, labels = batch
        logits = self.forward(images)
        preds, confs = self.postprocess(logits)
        correct = total = label_length = 0
        ned = confidence = 0.0
        for pred, conf_i, gt in zip(preds, confs, labels):
            confidence += conf_i
            pred = self.charset_adapter(pred)
            ned += edit_distance(pred, gt) / max(len(pred), len(gt), 1)
            correct += int(pred == gt)
            total += 1
            label_length += len(pred)
        return dict(output=BatchResult(total, correct, ned, confidence, label_length, None, None))

    def test_step(self, batch, batch_idx):
        return self._eval_step(batch, False)

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path: str, map_location="cpu", **kwargs):
        """Lightning .ckpt layout: {'hyper_parameters': ctor kwargs, 'state_dict': {'model.<key>': tensor}}."""
        ckpt = torch.load(checkpoint_path, map_location=map_location, weights_only=False)
        hp = dict(ckpt.get("hyper_parameters", {}))
        hp.update(kwargs)
        model = cls(**hp)
        sd = {k[len("model."):]: v for k, v in ckpt["state_dict"].items() if k.startswith("model.")}
        model.model.load_state_dict(sd)
        return model


class PARSeq(_System):
    def __init__(self, charset_train: str, charset_test: str, max_label_length: int, batch_size: int = 384,
                 lr: float = 7e-4, warmup_pct: float = 0.075, weight_decay: float = 0.0,
                 img_size: Sequence[int] = (32, 128), patch_size: Sequence[int] = (4, 8), embed_dim: int = 384,
                 enc_num_heads: int = 6, enc_mlp_ratio: int = 4, enc_depth: int = 12, dec_num_heads: int = 12,
                 dec_mlp_ratio: int = 4, dec_depth: int = 1, perm_num: int = 6, perm_forward: bool = True,
                 perm_mirrored: bool = True, decode_ar: bool = True, refine_iters: int = 1, dropout: float = 0.1,
                 **kwargs: Any) -> None:
        super().__init__()
        hp = dict(charset_train=charset_train, charset_test=charset_test, max_label_length=max_label_length,
                  batch_size=batch_size, lr=lr, warmup_pct=warmup_pct, weight_decay=weight_decay,
                  img_size=list(img_size), patch_size=list(patch_size), embed_dim=embed_dim,
                  enc_num_heads=enc_num_heads, enc_mlp_ratio=enc_mlp_ratio, enc_depth=enc_depth,
                  dec_num_heads=dec_num_heads, dec_mlp_ratio=dec_mlp_ratio, dec_depth=dec_depth, perm_num=perm_num,
                  perm_forward=perm_forward, perm_mirrored=perm_mirrored, decode_ar=decode_ar,
                  refine_iters=refine_iters, dropout=dropout)
        hp.update(kwargs)
        self.hparams = _HParams(**hp)
        self._init_base(charset_train, charset_test, batch_size, lr, warmup_pct, weight_decay)
        cfg = ParseqConfig(charset_train=charset_train, charset_test=charset_test, max_label_length=max_label_length,
                           img_size=tuple(img_size), patch_size=tuple(patch_size), embed_dim=embed_dim,
                           enc_num_heads=enc_num_heads, enc_mlp_ratio=enc_mlp_ratio, enc_depth=enc_depth,
                           dec_num_heads=dec_num_heads, dec_mlp_ratio=dec_mlp_ratio, dec_depth=dec_depth,
                           decode_ar=decode_ar, refine_iters=refine_iters, dropout=dropout,
                           name=str(kwargs.get("name", "parseq")))
        try:
            self.model = ParseqModel(cfg)
        except EngineError as e:  # pragma: no cover
            raise InvalidModelError(str(e)) from e

    def forward(self, images: Tensor, max_length: Optional[int] = None) -> Tensor:
        return self.model.forward(self.tokenizer, images, max_length)

    def forward_crops(self, crops, max_length: Optional[int] = None, rotation: int = 0) -> Tensor:
        """`forward` on variable-size RGB crops, resized on the GPU exactly as T.Resize(img_size, BICUBIC) does."""
        return self.model.forward_crops(self.tokenizer, crops, max_length, rotation)


class ViTSTR(_System):
    """Mirror of `strhub.models.vitstr.system.ViTSTR` (vitstr/system.py:29-71), inference side."""

    def __init__(self, charset_train: str, charset_test: str, max_label_length: int, batch_size: int = 384,
                 lr: float = 8.9e-4, warmup_pct: float = 0.075, weight_decay: float = 0.0,
                 img_size: Sequence[int] = (224, 224), patch_size: Sequence[int] = (16, 16), embed_dim: int = 384,
                 num_heads: int = 6, **kwargs: Any) -> None:
        super().__init__()
        hp = dict(charset_train=charset_train, charset_test=charset_test, max_label_length=max_label_length,
                  batch_size=batch_size, lr=lr, warmup_pct=warmup_pct, weight_decay=weight_decay,
                  img_size=list(img_size), patch_size=list(patch_size), embed_dim=embed_dim, num_heads=num_heads)
        hp.update(kwargs)
        self.hparams = _HParams(**hp)
        self._init_base(charset_train, charset_test, batch_size, lr, warmup_pct, weight_decay)
        self.max_label_length = max_label_length
        # depth=12, mlp_ratio=4, qkv_bias=True are fixed by the reference ctor (vitstr/system.py:50-59)
        cfg = ParseqConfig(charset_train=charset_train, charset_test=charset_test, max_label_length=max_label_length,
                           img_size=tuple(img_size), patch_size=tuple(patch_size), embed_dim=embed_dim,
                           enc_num_heads=num_heads, enc_mlp_ratio=4, enc_depth=12, arch="vitstr",
                           name=str(kwargs.get("name", "vitstr")))
        try:
            self.model = VitstrModel(cfg)
        except EngineError as e:  # pragma: no cover
            raise InvalidModelError(str(e)) from e

    def forward(self, images: Tensor, max_length: Optional[int] = None) -> Tensor:
        return self.model.forward_tokens(images, max_length)

    def forward_crops(self, crops, max_length: Optional[int] = None, rotation: int = 0) -> Tensor:
        """`forward` on variable-size RGB crops, resized on the GPU exactly as T.Resize(img_size, BICUBIC) does."""
        return self.model.forward_tokens_crops(crops, max_length, rotation)

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path: str, map_location="cpu", **kwargs):
        return super().load_from_checkpoint(checkpoint_path, map_location, **kwargs)

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        """Released ViTSTR weights are saved from the SYSTEM (strhub/models/utils.py:80-82: `m = model`), i.e. with a
        'model.' prefix; accept both layouts."""
        if all(k.startswith("model.") for k in state_dict):
            state_dict = {k[len("model."):]: v for k, v in state_dict.items()}
        return self.model.load_state_dict(state_dict, strict=strict, **kw)
